// pyin.cu -- probabilistic YIN (pYIN) on sm_100a: SURVEY 8(f) "next" row 2.
// Replaces librosa.pyin(y, fmin=60, fmax=500, sr=22050, hop_length=256) at
// /root/reference/spev_real_metrics.py:369 (and :311) -- the serial CPU bottleneck of the reference's
// cache build (seconds per utterance: YIN difference function, 100-threshold trough statistics and a
// 736-state Viterbi decode per utterance).
//
//   P1 k_yin_cmnd     frame -> cumulative-mean-normalised difference for lags min_period..max_period.
//                     d(tau) = e(0) + e(tau) - 2 acf(tau) with the autocorrelation summed directly
//                     (8-lag x 16-sample register tiles over even/odd float4 planes), energies from a
//                     block prefix sum, the reference's |.| < 1e-6 -> 0 clean-ups, block scan for the
//                     cumulative mean.
//   P2 k_pyin_observe frame -> troughs, parabolic refinement, for each of the 100 thresholds the
//                     Boltzmann prior over the troughs below it (bitmask + popcount ranks, float64),
//                     beta-weighted sum, global-minimum bonus, mapping to 10-cent pitch bins ->
//                     float32 log observation probabilities [F, n_bins] + voiced probability [F].
//   P3 k_pyin_viterbi utterance -> state path.  One CTA per utterance (dynamic work counter), one thread
//                     per pitch bin owning its voiced and unvoiced state, float64 log-domain recursion over
//                     the banded transition (kron(switch 2x2, triangular local band)); predecessors outside
//                     the band carry log(tiny) exactly as in the dense reference, so the best of them is the
//                     previous step's global maximum, found by a block arg-max.  Backpointers go to a
//                     caller-provided workspace; ties resolve to the lowest state index like np.argmax.
//   k_pitch_pool      per-phoneme masked mean / std of log-f0 from the decoded states (:399-414).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>
#include "spev_internal.cuh"
#include "tile_pipe.cuh"

struct spev_pyin {
    int device, sr;
    double fmin, fmax;
    int frame_length, win_length, hop, min_period, max_period, n_lags;
    int n_thresholds, n_bins, bins_per_semitone, trans_width;
    double no_trough_prob;
    double* d_thresholds;     // [n_thresholds+1]
    double* d_beta_probs;     // [n_thresholds]
    double* d_beta_cum;       // [n_thresholds+1] prefix sums of beta_probs (sequential, like np.sum of a slice... see note)
    double* d_boltz_exp;      // [kMaxTroughs] exp(-lambda k)
    double* d_boltz_fact;     // [kMaxTroughs+1] (1-exp(-lambda)) / (1-exp(-lambda N))
    double* d_ltrans;         // [n_classes][trans_width] x (stay, switch): log(t_switch * t_local + tiny)
    double* d_freqs;          // [n_bins]
    double* d_logf;           // [n_bins] log(freqs + 1e-8): the reference's f0_log on voiced frames (:399)
    int n_classes;
    std::vector<double> h_freqs, h_ltrans, h_beta;
};

namespace spev {

constexpr int kMaxTroughs = 192;          // 325 lags -> at most 163 local minima
constexpr int kMaskWords = kMaxTroughs / 32;
constexpr double kTiny64 = 2.2250738585072014e-308;
constexpr double kLogTiny64 = -708.3964185322641;   // log(DBL_MIN)

// ----------------------------------------------------------------------------------------------
// P1: cumulative mean normalised difference
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ float block_incl_scan(float v, float* s_w) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const float t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += t; }
    if (lane == 31) s_w[wid] = v;
    __syncthreads();
    if (wid == 0) {
        float w = lane < nw ? s_w[lane] : 0.f;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const float t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += t; }
        if (lane < nw) s_w[lane] = w;
    }
    __syncthreads();
    if (wid > 0) v += s_w[wid - 1];
    __syncthreads();
    return v;
}

// Block = 8 * O threads: O lag octets (lags 0 .. 8*O-1 >= max_period) x 8 segments of the 1024-sample window.
// The frame is staged twice: linearly (prefix sums) and split into even / odd float4 planes, so that the 8-lag x
// 16-sample register tile reads its 23 shifted samples with conflict-free LDS.128 (lane o needs float4 2*o + k of
// the linear order: stride 2 would be a 2-way bank conflict, planes make it stride 1).  128 FFMA per 10 LDS.128:
// 0.22 shared-memory wavefronts per FFMA -- the 4-lag tile of the first version (0.56) was shared-memory bound.
constexpr int kCmndSeg = 8;
__global__ void __launch_bounds__(512)
k_yin_cmnd(BatchView bv, const float* __restrict__ samples, float* __restrict__ yin, int frame_length, int win,
           int min_period, int max_period) {
    extern __shared__ __align__(16) float sm[];
    const int nthr = blockDim.x, O = nthr >> 3;
    float* s_z = sm;                                   // [2048] z[m] = frame sample m + 1 (sample 0 never contributes)
    float4* s_ev = reinterpret_cast<float4*>(sm + 2048);   // [256] float4 2n   of z
    float4* s_od = s_ev + 256 + 4;                         // [256] float4 2n+1 of z (+16 floats: the staging scatter of one
                                                           //       warp then covers all 32 banks instead of 16 twice)
    float* s_e = sm + 4096 + 16;                       // [2048] P[k] = sum_{m<k} z[m]^2
    float* s_part = s_e + 2048;                        // [8][nthr] partial autocorrelations
    float* s_w = s_part + kCmndSeg * nthr;             // [32]
    const int need = win + 8 * O;                      // z samples the tiles touch (<= frame_length - 1)
    const int n_lags = max_period - min_period + 1;
    const int64_t slots = static_cast<int64_t>(bv.n_ftiles) * kTileFrames;
    for (int64_t fidx = blockIdx.x; fidx < slots; fidx += gridDim.x) {
        const int64_t tile = fidx / kTileFrames;
        const spev_tile d = bv.ftiles[tile];
        const int fl = static_cast<int>(fidx - tile * kTileFrames);
        if (fl >= d.n) continue;                       // (uniform per CTA)
        // the frame_length window starts frame_length/2 before the frame centre; src0 is n_fft/2 before it; z skips sample 0
        const int64_t first = d.src0 - (frame_length / 2 - kNfft / 2) + static_cast<int64_t>(fl) * kHop + 1;
        __syncthreads();
        {
            const int i_lo = static_cast<int>(max(static_cast<int64_t>(0), min(static_cast<int64_t>(need), d.lo - first)));
            const int i_hi = static_cast<int>(max(static_cast<int64_t>(0), min(static_cast<int64_t>(need), d.hi - first)));
            const float* src = samples + first;
            float* ev = reinterpret_cast<float*>(s_ev);
            float* od = reinterpret_cast<float*>(s_od);
            for (int m = threadIdx.x; m < need; m += nthr) {
                const float v = (m >= i_lo && m < i_hi) ? __ldg(src + m) : 0.f;
                s_z[m] = v;
                ((m & 4) ? od : ev)[((m >> 3) << 2) | (m & 3)] = v;
            }
        }
        __syncthreads();
        {   // exclusive prefix sums of z^2 (numpy: cumsum in the input dtype): P[k], k = 0 .. need
            const int per = (need + nthr - 1) / nthr;
            const int b0 = min(need, threadIdx.x * per), b1 = min(need, b0 + per);
            float loc = 0.f;
            for (int i = b0; i < b1; ++i) loc = fmaf(s_z[i], s_z[i], loc);
            float run = block_incl_scan(loc, s_w) - loc;
            for (int i = b0; i < b1; ++i) { s_e[i] = run; run = fmaf(s_z[i], s_z[i], run); }
            if (b1 == need && b0 < need) s_e[need] = run;
        }
        {   // acf(tau) = sum_{m<W} z[m] z[m+tau]: thread = (lag octet o, window segment g), 8-lag x 16-sample register tile
            const int o = threadIdx.x % O, g = threadIdx.x / O;
            float c[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) c[r] = 0.f;
            const int n_begin = g * (win / 8 / kCmndSeg);          // float4-pair index: z index / 8
#pragma unroll 1
            for (int it = 0; it < win / 16 / kCmndSeg; ++it) {
                const int n = n_begin + 2 * it;
                float A[16], B[24];
                *reinterpret_cast<float4*>(A) = s_ev[n];       *reinterpret_cast<float4*>(A + 4) = s_od[n];
                *reinterpret_cast<float4*>(A + 8) = s_ev[n + 1]; *reinterpret_cast<float4*>(A + 12) = s_od[n + 1];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    *reinterpret_cast<float4*>(B + 8 * k) = s_ev[n + o + k];
                    *reinterpret_cast<float4*>(B + 8 * k + 4) = s_od[n + o + k];
                }
#pragma unroll
                for (int m = 0; m < 16; ++m)
#pragma unroll
                    for (int r = 0; r < 8; ++r) c[r] = fmaf(A[m], B[m + r], c[r]);
            }
            float* dst = s_part + g * nthr + 8 * o;
            *reinterpret_cast<float4*>(dst) = make_float4(c[0], c[1], c[2], c[3]);
            *reinterpret_cast<float4*>(dst + 4) = make_float4(c[4], c[5], c[6], c[7]);
        }
        __syncthreads();
        const int tau = threadIdx.x;                    // one lag per thread from here on
        float dval = 0.f;
        if (tau >= 1 && tau <= max_period) {
            float p[kCmndSeg];
#pragma unroll
            for (int k = 0; k < kCmndSeg; ++k) p[k] = s_part[k * nthr + tau];
            float acf = ((p[0] + p[1]) + (p[2] + p[3])) + ((p[4] + p[5]) + (p[6] + p[7]));
            float e_tau = s_e[tau + win] - s_e[tau];    // samples tau+1 .. tau+W of the frame
            float e_0 = s_e[win] - s_e[0];
            if (fabsf(acf) < 1e-6f) acf = 0.f;          // the reference's clean-ups
            if (fabsf(e_tau) < 1e-6f) e_tau = 0.f;
            if (fabsf(e_0) < 1e-6f) e_0 = 0.f;
            dval = e_0 + e_tau - 2.f * acf;
        }
        const float cum = block_incl_scan(dval, s_w);   // sum of d(1..tau)
        if (tau >= min_period && tau <= max_period) {
            const float cm = cum / static_cast<float>(tau);
            yin[(d.row0 + fl) * n_lags + (tau - min_period)] = dval / (cm + 1.17549435e-38f);
        }
    }
}

// ----------------------------------------------------------------------------------------------
// P1 (round 2): the same curve from SHARED partial sums.
// Consecutive frames overlap by 75 % (hop 256, window 1024): the autocorrelation of frame f is the sum of eight
// 128-sample segment partials  S[s](tau) = sum_{m in segment s} z[m] z[m + tau],  s = 2f .. 2f + 7, and a segment is
// shared by the four frames that cover it.  k_yin_cmnd above recomputes every segment for each of them (393 k FMA
// per frame); here a CTA takes a run of up to 16 consecutive frames of one item, computes its 2*16 + 6 = 38 segment
// partials ONCE (the same 8-lag x 16-sample register tile, the same summation order) and every frame adds its eight
// in the same pairwise order -- bit-identical autocorrelations for 2.4 instead of 8 segments per frame.  The per-frame
// rest (energy prefix sums, differences, cumulative mean) is one warp per frame, no CTA barrier.
// ----------------------------------------------------------------------------------------------
constexpr int kCmndGroup = 16;                         // frames per pass = warps per CTA
constexpr int kCmndThreads = kCmndGroup * 32;
__global__ void __launch_bounds__(kCmndThreads)
k_yin_cmnd_shared(BatchView bv, const float* __restrict__ samples, float* __restrict__ yin, int frame_length, int win,
                  int min_period, int max_period, int O /* lag octets: lags 0 .. 8*O-1 */) {
    extern __shared__ __align__(16) float sm[];
    const int L8 = 8 * O;                               // lags held per segment
    const int need = win + L8;                          // z samples one frame touches
    const int zmax = (kCmndGroup - 1) * kHop + need;    // z samples of a full group
    const int nplane = (zmax + 7) / 8 + 4;              // float4 per plane (+ slack for the 24-sample B reads)
    float* s_z = sm;                                                     // [zmax] linear (prefix sums)
    float4* s_ev = reinterpret_cast<float4*>(sm + ((zmax + 3) & ~3));    // float4 2n   of z
    float4* s_od = s_ev + nplane + 4;                                    // float4 2n+1 of z (bank offset, see above)
    float* s_part = reinterpret_cast<float*>(s_od + nplane);             // [2*G + 6][L8] segment partials
    float* s_e = s_part + (2 * kCmndGroup + 6) * L8;                     // [G][need + 1] per-frame prefix sums of z^2
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_lags = max_period - min_period + 1;
    const int per_tile = (kTileFrames + kCmndGroup - 1) / kCmndGroup;
    const int64_t n_groups = static_cast<int64_t>(bv.n_ftiles) * per_tile;
    for (int64_t gi = blockIdx.x; gi < n_groups; gi += gridDim.x) {
        const spev_tile d = bv.ftiles[gi / per_tile];
        const int f0 = static_cast<int>(gi % per_tile) * kCmndGroup;
        const int ng = min(kCmndGroup, d.n - f0);
        if (ng <= 0) continue;                          // (uniform per CTA)
        const int nseg = 2 * (ng - 1) + 8;
        const int count = (ng - 1) * kHop + need;
        // the frame_length window starts frame_length/2 before the frame centre; src0 is n_fft/2 before it; z skips sample 0
        const int64_t first = d.src0 - (frame_length / 2 - kNfft / 2) + static_cast<int64_t>(f0) * kHop + 1;
        __syncthreads();
        {
            const int i_lo = static_cast<int>(max(static_cast<int64_t>(0), min(static_cast<int64_t>(count), d.lo - first)));
            const int i_hi = static_cast<int>(max(static_cast<int64_t>(0), min(static_cast<int64_t>(count), d.hi - first)));
            const float* src = samples + first;
            float* ev = reinterpret_cast<float*>(s_ev);
            float* od = reinterpret_cast<float*>(s_od);
            for (int m = threadIdx.x; m < count + 32; m += blockDim.x) {      // + 32: the B tiles read a little past `count`
                const float v = (m >= i_lo && m < i_hi) ? __ldg(src + m) : 0.f;
                if (m < zmax) s_z[m] = v;
                if ((m >> 3) < nplane) ((m & 4) ? od : ev)[((m >> 3) << 2) | (m & 3)] = v;
            }
        }
        __syncthreads();
        // ---- segment partials: work item = (segment, lag octet), 8-lag x 16-sample register tile ----
        for (int w = threadIdx.x; w < nseg * O; w += blockDim.x) {
            const int sg = w / O, o = w - sg * O;
            float c[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) c[r] = 0.f;
            const int n_begin = sg * 16;                // float4-pair index of the segment's first sample
#pragma unroll 1
            for (int it = 0; it < 8; ++it) {
                const int n = n_begin + 2 * it;
                float A[16], B[24];
                *reinterpret_cast<float4*>(A) = s_ev[n];       *reinterpret_cast<float4*>(A + 4) = s_od[n];
                *reinterpret_cast<float4*>(A + 8) = s_ev[n + 1]; *reinterpret_cast<float4*>(A + 12) = s_od[n + 1];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    *reinterpret_cast<float4*>(B + 8 * k) = s_ev[n + o + k];
                    *reinterpret_cast<float4*>(B + 8 * k + 4) = s_od[n + o + k];
                }
#pragma unroll
                for (int m = 0; m < 16; ++m)
#pragma unroll
                    for (int r = 0; r < 8; ++r) c[r] = fmaf(A[m], B[m + r], c[r]);
            }
            float* dst = s_part + sg * L8 + 8 * o;
            *reinterpret_cast<float4*>(dst) = make_float4(c[0], c[1], c[2], c[3]);
            *reinterpret_cast<float4*>(dst + 4) = make_float4(c[4], c[5], c[6], c[7]);
        }
        // ---- per-frame prefix sums of z^2 (numpy: cumsum in the input dtype), one warp per frame ----
        if (warp < ng) {
            const float* z = s_z + warp * kHop;
            float* e = s_e + warp * (need + 1);
            const int per = (need + 31) / 32;
            const int b0 = min(need, lane * per), b1 = min(need, b0 + per);
            float loc = 0.f;
            for (int i = b0; i < b1; ++i) loc = fmaf(z[i], z[i], loc);
            float run = loc;
#pragma unroll
            for (int o2 = 1; o2 < 32; o2 <<= 1) { const float t = __shfl_up_sync(0xffffffffu, run, o2); if (lane >= o2) run += t; }
            run -= loc;                                  // exclusive
            for (int i = b0; i < b1; ++i) { e[i] = run; run = fmaf(z[i], z[i], run); }
            if (b1 == need && b0 < need) e[need] = run;
        }
        __syncthreads();
        // ---- difference function, cumulative mean normalisation: one warp per frame, lags in chunks of 32 ----
        if (warp < ng) {
            const float* e = s_e + warp * (need + 1);
            const float* part = s_part + (2 * warp) * L8;
            float carry = 0.f;
            float e_0 = e[win] - e[0];
            if (fabsf(e_0) < 1e-6f) e_0 = 0.f;
            float* out = yin + (d.row0 + f0 + warp) * n_lags;
            for (int t0 = 0; t0 <= max_period; t0 += 32) {
                const int tau = t0 + lane;
                float dval = 0.f;
                if (tau >= 1 && tau <= max_period) {
                    float p[kCmndSeg];
#pragma unroll
                    for (int k = 0; k < kCmndSeg; ++k) p[k] = part[k * L8 + tau];
                    float acf = ((p[0] + p[1]) + (p[2] + p[3])) + ((p[4] + p[5]) + (p[6] + p[7]));
                    float e_tau = e[tau + win] - e[tau];    // samples tau+1 .. tau+W of the frame
                    if (fabsf(acf) < 1e-6f) acf = 0.f;      // the reference's clean-ups
                    if (fabsf(e_tau) < 1e-6f) e_tau = 0.f;
                    dval = e_0 + e_tau - 2.f * acf;
                }
                float cum = dval;
#pragma unroll
                for (int o2 = 1; o2 < 32; o2 <<= 1) { const float t = __shfl_up_sync(0xffffffffu, cum, o2); if (lane >= o2) cum += t; }
                cum += carry;                               // sum of d(1..tau)
                carry = __shfl_sync(0xffffffffu, cum, 31);
                if (tau >= min_period && tau <= max_period) {
                    const float cm = cum / static_cast<float>(tau);
                    out[tau - min_period] = dval / (cm + 1.17549435e-38f);
                }
            }
        }
    }
}

// ----------------------------------------------------------------------------------------------
// P2: observation probabilities
// ----------------------------------------------------------------------------------------------
struct ObsParams {
    int n_lags, min_period, n_thresholds, n_bins, bins_per_semitone, sr;
    double fmin, no_trough_prob;
    const double* thresholds;
    const double* beta_probs;
    const double* beta_cum;
    const double* boltz_exp;
    const double* boltz_fact;
};

constexpr int kObsThreads = 128;
__global__ void __launch_bounds__(kObsThreads)
k_pyin_observe(const float* __restrict__ yin, int64_t n_frames, ObsParams p, float* __restrict__ logobs,
               float* __restrict__ log_unvoiced, float* __restrict__ voiced_prob) {
    __shared__ float s_y[512];
    __shared__ int s_tidx[kMaxTroughs];
    __shared__ int s_ithr[kMaxTroughs];
    __shared__ double s_prob[kMaxTroughs];
    __shared__ unsigned s_mask[128][kMaskWords];     // [threshold][word]: troughs below that threshold
    __shared__ int s_count[128];
    __shared__ unsigned s_cmask[128][kMaskWords];    // the same at the change points only, prefix-ORed
    __shared__ int s_cp[128], s_cpidx[128];
    __shared__ double s_cw[128];
    __shared__ int s_wcnt[kObsThreads / 32];
    __shared__ double s_wsum[kObsThreads / 32];
    __shared__ double s_obs[512];
    __shared__ double s_thr[104], s_beta[104], s_bcum[104], s_bexp[kMaxTroughs], s_bfact[kMaxTroughs + 1];
    const int L = p.n_lags, NT = p.n_thresholds;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int i = threadIdx.x; i <= NT; i += blockDim.x) { s_thr[i] = p.thresholds[i]; s_bcum[i] = p.beta_cum[i]; }
    for (int i = threadIdx.x; i < NT; i += blockDim.x) s_beta[i] = p.beta_probs[i];
    for (int i = threadIdx.x; i < kMaxTroughs; i += blockDim.x) { s_bexp[i] = p.boltz_exp[i]; s_bfact[i + 1] = p.boltz_fact[i + 1]; }
    const float log_tiny_f = static_cast<float>(kLogTiny64);
    for (int64_t f = blockIdx.x; f < n_frames; f += gridDim.x) {
        __syncthreads();
        for (int i = threadIdx.x; i < L; i += blockDim.x) s_y[i] = yin[f * L + i];
        for (int i = threadIdx.x; i < p.n_bins; i += blockDim.x) s_obs[i] = 0.0;
        for (int i = threadIdx.x; i < NT * kMaskWords; i += blockDim.x) (&s_mask[0][0])[i] = 0u;
        __syncthreads();
        // troughs: localmin (x[i] < x[i-1] && x[i] <= x[i+1], edge-padded); first element: x[0] < x[1].
        // ordered compaction, kObsThreads lags per round
        int K = 0;
        for (int base = 0; base < L; base += kObsThreads) {
            const int i = base + threadIdx.x;
            bool tr = false;
            if (i < L) {
                const float c = s_y[i];
                if (i == 0) tr = L > 1 && c < s_y[1];
                else tr = (c < s_y[i - 1]) && (c <= (i + 1 < L ? s_y[i + 1] : c));
            }
            const unsigned bal = __ballot_sync(0xffffffffu, tr);
            if (lane == 0) s_wcnt[wid] = __popc(bal);
            __syncthreads();
            int off = K;
            for (int w = 0; w < wid; ++w) off += s_wcnt[w];
            if (tr) { const int k = off + __popc(bal & ((1u << lane) - 1u)); if (k < kMaxTroughs) s_tidx[k] = i; }
            for (int w = 0; w < kObsThreads / 32; ++w) K += s_wcnt[w];
            __syncthreads();
        }
        K = min(K, kMaxTroughs);
        if (K == 0) {                                    // (uniform) no trough: all mass on the unvoiced states
            if (threadIdx.x == 0) {
                voiced_prob[f] = 0.f;
                log_unvoiced[f] = static_cast<float>(log(1.0 / p.n_bins + kTiny64));
            }
            for (int i = threadIdx.x; i < p.n_bins; i += blockDim.x) logobs[f * p.n_bins + i] = log_tiny_f;
            continue;
        }
        // first threshold index each trough lies below (thresholds[i+1] > h); NT if none
        for (int k = threadIdx.x; k < K; k += blockDim.x) {
            const double h = static_cast<double>(s_y[s_tidx[k]]);
            int lo = 0, hi = NT;
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (h < s_thr[mid + 1]) hi = mid; else lo = mid + 1; }
            s_ithr[k] = lo;
            if (lo < NT) atomicOr(&s_mask[lo][k >> 5], 1u << (k & 31));
        }
        __syncthreads();
        // The set of troughs below threshold i only changes at the thresholds some trough starts at ("change
        // points", at most min(K, 100) of them): compact them, so that the sums below run over runs of equal
        // Boltzmann terms weighted by the beta mass of the run instead of over all 100 thresholds.
        int J = 0;
        {
            const int i = threadIdx.x;                   // NT <= blockDim.x
            bool cp = false;
            if (i < NT) {
#pragma unroll
                for (int w = 0; w < kMaskWords; ++w) cp |= s_mask[i][w] != 0u;
            }
            const unsigned bal = __ballot_sync(0xffffffffu, cp);
            if (lane == 0) s_wcnt[wid] = __popc(bal);
            __syncthreads();
            int off = 0;
            for (int w = 0; w < wid; ++w) off += s_wcnt[w];
            for (int w = 0; w < kObsThreads / 32; ++w) J += s_wcnt[w];
            if (cp) {
                const int j = off + __popc(bal & ((1u << lane) - 1u));
                s_cp[j] = i;
                s_cpidx[i] = j;
#pragma unroll
                for (int w = 0; w < kMaskWords; ++w) s_cmask[j][w] = s_mask[i][w];
            }
        }
        __syncthreads();
        if (threadIdx.x < kMaskWords) {                 // prefix-OR over the change points
            unsigned run = 0u;
            for (int j = 0; j < J; ++j) { run |= s_cmask[j][threadIdx.x]; s_cmask[j][threadIdx.x] = run; }
        }
        __syncthreads();
        for (int j = threadIdx.x; j < J; j += blockDim.x) {
            int c = 0;
#pragma unroll
            for (int w = 0; w < kMaskWords; ++w) c += __popc(s_cmask[j][w]);
            s_count[j] = c;
            s_cw[j] = s_bcum[j + 1 < J ? s_cp[j + 1] : NT] - s_bcum[s_cp[j]];   // beta mass of thresholds [cp_j, cp_j+1)
        }
        __syncthreads();
        // probs[k] = sum_i boltzmann.pmf(rank_{k,i}, lambda, n_i) * beta_probs[i]   (i >= ithr[k]);
        // four threads per trough (change points interleaved), partials combined in a fixed order
        for (int kb = 0; kb < K; kb += kObsThreads / 4) {
            const int k = kb + (threadIdx.x >> 2), sub = threadIdx.x & 3;
            double acc = 0.0;
            if (k < K && s_ithr[k] < NT) {
                const int w0 = k >> 5;
                const unsigned below = (1u << (k & 31)) - 1u;
                for (int j = s_cpidx[s_ithr[k]] + sub; j < J; j += 4) {
                    int rank = __popc(s_cmask[j][w0] & below);
                    for (int w = 0; w < w0; ++w) rank += __popc(s_cmask[j][w]);
                    acc += (s_bfact[s_count[j]] * s_bexp[rank]) * s_cw[j];
                }
            }
            acc += __shfl_xor_sync(0xffffffffu, acc, 1);
            acc += __shfl_xor_sync(0xffffffffu, acc, 2);
            if (k < K && sub == 0) s_prob[k] = acc;
        }
        __syncthreads();
        {   // global minimum bonus (np.argmin: first minimum) -- warp 0 arg-min over the trough heights
            if (wid == 0) {
                float hmin = INFINITY;
                int gm = 0x7fffffff;
                for (int k = lane; k < K; k += 32) { const float h = s_y[s_tidx[k]]; if (h < hmin) { hmin = h; gm = k; } }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const float oh = __shfl_xor_sync(0xffffffffu, hmin, o);
                    const int og = __shfl_xor_sync(0xffffffffu, gm, o);
                    if (oh < hmin || (oh == hmin && og < gm)) { hmin = oh; gm = og; }
                }
                if (lane == 0) s_prob[gm] += p.no_trough_prob * s_bcum[s_ithr[gm]];
            }
        }
        __syncthreads();
        // candidates -> pitch bins, one thread per trough.  numpy assigns in ascending lag order, so of several
        // troughs landing in one bin the LAST non-zero one stays: a trough writes unless a later one claims its bin.
        for (int k = threadIdx.x; k < K; k += blockDim.x) {
            // librosa's CMND array is float64 even for float32 audio (the cumulative mean divides by an int64 lag
            // vector), so the probabilities and the parabolic refinement below are float64 on the stored values
            const double pr = s_prob[k];
            int bin = -1;
            if (pr != 0.0) {                                    // np.nonzero
                const int i = s_tidx[k];
                double shift = 0.0;
                if (i >= 1 && i + 1 < L) {
                    const double y0 = s_y[i - 1], y1 = s_y[i], y2 = s_y[i + 1];
                    const double a = y2 + y0 - 2.0 * y1;
                    const double b = (y2 - y0) / 2.0;
                    if (fabs(b) < fabs(a)) shift = -b / a;
                }
                const double period = static_cast<double>(p.min_period + i) + shift;
                const double f0 = static_cast<double>(p.sr) / period;
                double bi = rint(12.0 * p.bins_per_semitone * log2(f0 / p.fmin));
                bi = fmin(fmax(bi, 0.0), static_cast<double>(p.n_bins));
                bin = static_cast<int>(bi);
                if (bin >= p.n_bins) bin = -1;                  // bin == n_bins falls in the unvoiced half, overwritten there
            }
            s_ithr[k] = bin;                                    // (the threshold indices are dead from here on)
        }
        __syncthreads();
        for (int k = threadIdx.x; k < K; k += blockDim.x) {
            const int bin = s_ithr[k];
            if (bin < 0) continue;
            bool last = true;
            for (int k2 = k + 1; k2 < K; ++k2) if (s_ithr[k2] == bin) { last = false; break; }
            if (last) s_obs[bin] = s_prob[k];
        }
        __syncthreads();
        {   // voiced probability = clip(sum of the voiced bins, 0, 1)
            double part = 0.0;
            for (int i = threadIdx.x; i < p.n_bins; i += blockDim.x) part += s_obs[i];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
            if (lane == 0) s_wsum[wid] = part;
            __syncthreads();
            if (threadIdx.x == 0) {
                double vsum = (s_wsum[0] + s_wsum[1]) + (s_wsum[2] + s_wsum[3]);
                vsum = fmin(fmax(vsum, 0.0), 1.0);
                voiced_prob[f] = static_cast<float>(vsum);
                log_unvoiced[f] = static_cast<float>(log((1.0 - vsum) / p.n_bins + kTiny64));
            }
        }
        for (int i = threadIdx.x; i < p.n_bins; i += blockDim.x) {
            const double o = s_obs[i];
            logobs[f * p.n_bins + i] = o == 0.0 ? log_tiny_f : static_cast<float>(log(o + kTiny64));
        }
    }
}

// ----------------------------------------------------------------------------------------------
// P3: Viterbi
// ----------------------------------------------------------------------------------------------
struct VitParams {
    int n_bins, width, n_classes;
    const double2* tab;       // [n_classes][width] (stay, switch) log transition probabilities
};

#ifndef SPEV_VIT_CTAS
#define SPEV_VIT_CTAS 2   // 3 (56 registers) was measured: 28.4 ms either way -- the kernel is ALU / FP64-pipe bound, not latency bound
#endif
constexpr int kVitThreads = 384;                 // one thread per pitch bin: it owns the voiced AND the unvoiced state of that bin
struct ArgMax { double v; int i; };
__device__ __forceinline__ ArgMax warp_argmax(ArgMax a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, a.v, o);
        const int oi = __shfl_xor_sync(0xffffffffu, a.i, o);
        if (ov > a.v || (ov == a.v && oi < a.i)) { a.v = ov; a.i = oi; }
    }
    return a;
}

// (ptxas turns this into DSETP + 2 FSEL + SEL whether it is written as a branch, a select or predicated PTX moves:
// 12 of the ~23 instructions per candidate sit on the ALU pipe, which is what bounds the kernel.)
__device__ __forceinline__ void upd_max(double& m, int& a, double s, int i) {
    if (s > m) { m = s; a = i; }
}

// Transition table as the kernel reads it: tab[cls][d] = (log P(stay in the voicing half), log P(switch half)) for a
// predecessor of row class cls and bin offset d - half.  kron(switch, local) gives the same value for
// voiced->voiced and unvoiced->unvoiced (and for the two switches), so two numbers serve all four (vp, v) pairs.
template <bool LT_SMEM>
__global__ void __launch_bounds__(kVitThreads, SPEV_VIT_CTAS)
k_pyin_viterbi(const float* __restrict__ logobs, const float* __restrict__ log_unvoiced,
               const int64_t* __restrict__ frame_off, int n_items, VitParams p, unsigned short* __restrict__ ptr,
               int* __restrict__ states, unsigned* __restrict__ work_counter) {
    extern __shared__ __align__(16) double smd[];
    double2* s_val = reinterpret_cast<double2*>(smd);      // [2][n_bins]: (voiced, unvoiced) value of each bin
    double2* s_tab = s_val + 2 * p.n_bins;                 // [n_classes][width] when LT_SMEM
    __shared__ double s_red_v[2 * (kVitThreads / 32)];
    __shared__ int s_red_i[2 * (kVitThreads / 32)];
    __shared__ int s_item;
    const int nb = p.n_bins, S = 2 * nb, W = p.width, half = W / 2;
    if (LT_SMEM) for (int i = threadIdx.x; i < p.n_classes * W; i += blockDim.x) s_tab[i] = p.tab[i];
    const double2* tab = LT_SMEM ? s_tab : p.tab;          // wide bands (hop 512) stay in global memory / L1
    const int b = threadIdx.x;
    const bool act = b < nb;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int blo = max(0, b - half), bhi = min(nb - 1, b + half);
    // predecessor rows by class: [blo, e1) left edge (class = row), [e1, e2) interior (class = half), [e2, bhi] right edge
    const int e1 = min(bhi + 1, max(blo, half)), e2 = max(e1, min(bhi + 1, nb - half));
    const double log_init_unv = log(1.0 / nb + kTiny64);

    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_item = static_cast<int>(atomicAdd(work_counter, 1u));
        __syncthreads();
        const int u = s_item;
        if (u >= n_items) break;
        const int64_t f0 = frame_off[u];
        const int T = static_cast<int>(frame_off[u + 1] - f0);
        if (T <= 0) continue;
        // t = 0: log_prob[0] + log(p_init): p_init = 0 on voiced states, 1/n_bins on unvoiced ones
        double cur0 = -INFINITY, cur1 = -INFINITY;
        if (act) {
            cur0 = static_cast<double>(logobs[f0 * nb + b]) + kLogTiny64;
            cur1 = static_cast<double>(log_unvoiced[f0]) + log_init_unv;
            s_val[b] = make_double2(cur0, cur1);
        }
        for (int t = 1; t < T; ++t) {
            const int64_t ft = f0 + t;
            // this step's observations (issued early: the loads overlap the arg-max reduction)
            const float lp0f = act ? logobs[ft * nb + b] : 0.f;
            const float lp1f = log_unvoiced[ft];
            // block arg-max of the previous values (lowest state index on ties)
            ArgMax m;
            if (act) { if (cur1 > cur0) { m.v = cur1; m.i = nb + b; } else { m.v = cur0; m.i = b; } }
            else { m.v = -INFINITY; m.i = 0x7fffffff; }
            m = warp_argmax(m);
            double* red_v = s_red_v + (t & 1) * (kVitThreads / 32);     // double-buffered: one barrier per step
            int* red_i = s_red_i + (t & 1) * (kVitThreads / 32);
            if (lane == 0) { red_v[wid] = m.v; red_i[wid] = m.i; }
            __syncthreads();                               // also publishes s_val[prev]
            // every warp finishes the reduction for itself (no second barrier, no serial section)
            if (lane < kVitThreads / 32) { m.v = red_v[lane]; m.i = red_i[lane]; }
            else { m.v = -INFINITY; m.i = 0x7fffffff; }
            m = warp_argmax(m);
            const double gmax = m.v;
            const int garg = m.i;
            const double2* prev = s_val + ((t - 1) & 1) * nb;
            double2* next = s_val + (t & 1) * nb;
            if (act) {
                // four independent running maxima: (from voiced | unvoiced) x (to voiced | unvoiced), ascending bin
                double m00 = -INFINITY, m01 = -INFINITY, m10 = -INFINITY, m11 = -INFINITY;
                int a00 = 0, a01 = 0, a10 = 0, a11 = 0;
                auto cand = [&](int bp, const double2 ab) {
                    const double2 x = prev[bp];
                    const double s00 = x.x + ab.x, s01 = x.x + ab.y, s10 = x.y + ab.y, s11 = x.y + ab.x;
                    upd_max(m00, a00, s00, bp);
                    upd_max(m01, a01, s01, bp);
                    upd_max(m10, a10, s10, bp);
                    upd_max(m11, a11, s11, bp);
                };
                for (int bp = blo; bp < e1; ++bp) cand(bp, tab[bp * W + (b - bp + half)]);
                {
                    const double2* q = tab + half * W + (b - e1 + half);
#pragma unroll 2
                    for (int bp = e1; bp < e2; ++bp, --q) cand(bp, *q);
                }
                for (int bp = e2; bp <= bhi; ++bp) cand(bp, tab[(half + 1 + bp - (nb - half)) * W + (b - bp + half)]);
                // merge the two source halves; the voiced half holds the lower state indices and wins ties
                double best0 = m00, best1 = m01;
                int arg0 = a00, arg1 = a01;
                if (m10 > best0) { best0 = m10; arg0 = nb + a10; }
                if (m11 > best1) { best1 = m11; arg1 = nb + a11; }
                // predecessors outside the band have transition probability 0 -> log(0 + tiny); the best
                // of them is the global maximum when that state is itself outside the band
                const int ga = garg;
                const int gb = ga >= nb ? ga - nb : ga;
                if (gb < blo || gb > bhi) {
                    const double sc = gmax + kLogTiny64;
                    if (sc > best0 || (sc == best0 && ga < arg0)) { best0 = sc; arg0 = ga; }
                    if (sc > best1 || (sc == best1 && ga < arg1)) { best1 = sc; arg1 = ga; }
                }
                cur0 = static_cast<double>(lp0f) + best0;
                cur1 = static_cast<double>(lp1f) + best1;
                next[b] = make_double2(cur0, cur1);
                ptr[ft * S + b] = static_cast<unsigned short>(arg0);
                ptr[ft * S + nb + b] = static_cast<unsigned short>(arg1);
            }
            // (the __syncthreads at the top of the next iteration orders next[] before it is read)
        }
        // final arg-max and backtrace
        __syncthreads();                                   // the last step's reduction buffers are no longer read
        {
            ArgMax m;
            if (act) { if (cur1 > cur0) { m.v = cur1; m.i = nb + b; } else { m.v = cur0; m.i = b; } }
            else { m.v = -INFINITY; m.i = 0x7fffffff; }
            m = warp_argmax(m);
            if (lane == 0) { s_red_v[wid] = m.v; s_red_i[wid] = m.i; }
            __syncthreads();
            if (threadIdx.x == 0) {
                double bv = -INFINITY;
                int bi = 0x7fffffff;
                for (int w = 0; w < kVitThreads / 32; ++w)
                    if (s_red_v[w] > bv || (s_red_v[w] == bv && s_red_i[w] < bi)) { bv = s_red_v[w]; bi = s_red_i[w]; }
                int st = bi;
                states[f0 + T - 1] = st;
                for (int t = T - 2; t >= 0; --t) {
                    st = ptr[(f0 + t + 1) * S + st];
                    states[f0 + t] = st;
                }
            }
        }
    }
}

__global__ void k_pyin_finish(const int* __restrict__ states, int64_t n, int n_bins, const double* __restrict__ freqs,
                              float* __restrict__ f0, unsigned char* __restrict__ voiced) {
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int s = states[i];
        const bool vflag = s < n_bins;
        if (voiced) voiced[i] = vflag ? 1 : 0;
        if (f0) f0[i] = vflag ? static_cast<float>(freqs[s % n_bins]) : __int_as_float(0x7fc00000);
    }
}

// ---- per-phoneme pitch statistics (spev_real_metrics.py:399-414) -----------------------------------
// f0_log = log(f0 + 1e-8) on voiced frames (unvoiced ones are log(2e-8) < -5 and masked out there):
//   pitch = clip((mean(voiced f0_log) - p_mean) / p_std, lo, hi)   or clip(0) when the phone has no voiced frame
//   rough = clip(std(voiced f0_log), 0, rough_hi)                  (np.std: population), 0 without voiced frames
// One warp per utterance (warp scan of the durations), one lane per phoneme, float64 like numpy.
__global__ void k_pitch_pool(const int* __restrict__ states, const int64_t* __restrict__ frame_off,
                             const long long* __restrict__ durs, const int64_t* __restrict__ phone_off, int U, int n_bins,
                             const double* __restrict__ logf, double p_mean, double p_std, float lo, float hi,
                             float rough_hi, float* __restrict__ pitch, float* __restrict__ rough) {
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    for (int u = blockIdx.x * wpb + (threadIdx.x >> 5); u < U; u += gridDim.x * wpb) {
        const int64_t p0 = phone_off[u], p1 = phone_off[u + 1];
        const int* st = states + frame_off[u];
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
                const long long end = min(static_cast<long long>(T), start + dd);
                double sum = 0.0;
                int n = 0;
                for (long long t = start; t < end; ++t) { const int s = st[t]; if (s < n_bins) { sum += logf[s]; ++n; } }
                double pv = 0.0, rv = 0.0;
                if (n > 0) {
                    const double mean = sum / n;
                    double ss = 0.0;
                    for (long long t = start; t < end; ++t) { const int s = st[t]; if (s < n_bins) { const double dlt = logf[s] - mean; ss += dlt * dlt; } }
                    pv = (mean - p_mean) / p_std;
                    rv = sqrt(ss / n);
                }
                pitch[p] = static_cast<float>(fmin(fmax(pv, static_cast<double>(lo)), static_cast<double>(hi)));
                rough[p] = static_cast<float>(fmin(fmax(rv, 0.0), static_cast<double>(rough_hi)));
            }
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
    }
}

}  // namespace spev

using namespace spev;

// ----------------------------------------------------------------------------------------------
// host side: tables (restating librosa.pyin's set-up) and the C ABI
// ----------------------------------------------------------------------------------------------
static double beta_cdf_int(double x, int a, int b) {
    // I_x(a, b) for integer a, b = 1 - sum_{j<a} C(n, j) x^j (1-x)^(n-j), n = a+b-1 (the short, accurate side)
    const int n = a + b - 1;
    double s = 0.0;
    const bool upper = x >= 0.25;                          // sum the side with the smaller total
    for (int j = upper ? 0 : a; j <= (upper ? a - 1 : n); ++j) {
        double c = 1.0;
        for (int q = 1; q <= j; ++q) c = c * (n - j + q) / q;
        s += c * std::pow(x, j) * std::pow(1.0 - x, n - j);
    }
    return upper ? 1.0 - s : s;
}

extern "C" {

int spev_pyin_create(spev_pyin** out, int device, int sr, int hop_length, float fmin, float fmax,
                     const double* beta_probs_host) {
    SPEV_REQUIRE(out, SPEV_E_INVALID, "spev_pyin_create: out is null");
    *out = nullptr;
    SPEV_REQUIRE(sr > 0 && fmin > 0.f && fmax > fmin, SPEV_E_INVALID, "spev_pyin_create: need sr > 0, 0 < fmin < fmax");
    SPEV_REQUIRE(hop_length > 0 && hop_length % kHop == 0, SPEV_E_UNSUPPORTED,
                 "spev_pyin_create: hop_length must be a multiple of 256 (frames are taken from the hop-256 grid)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("spev_pyin_create: no CUDA device (this library has no CPU fallback)");
        return SPEV_E_DEVICE;
    }
    SPEV_REQUIRE(device >= 0 && device < ndev, SPEV_E_DEVICE, "spev_pyin_create: device out of range");
    SPEV_CUDA(cudaSetDevice(device));
    spev_pyin* c = new spev_pyin();
    c->device = device; c->sr = sr; c->fmin = fmin; c->fmax = fmax;
    c->frame_length = 2048; c->win_length = 1024; c->hop = hop_length;
    c->min_period = static_cast<int>(std::floor(static_cast<double>(sr) / fmax));
    c->max_period = std::min(static_cast<int>(std::ceil(static_cast<double>(sr) / fmin)), c->frame_length - c->win_length - 1);
    c->n_lags = c->max_period - c->min_period + 1;
    c->n_thresholds = 100; c->no_trough_prob = 0.01;
    c->bins_per_semitone = 10;                                     // ceil(1 / resolution), resolution = 0.1
    c->n_bins = static_cast<int>(std::floor(12.0 * c->bins_per_semitone * std::log2(static_cast<double>(fmax) / fmin))) + 1;
    const int max_semitones = static_cast<int>(std::nearbyint(35.92 * 12.0 * c->hop / sr));
    c->trans_width = max_semitones * c->bins_per_semitone + 1;
    c->d_thresholds = c->d_beta_probs = c->d_beta_cum = c->d_boltz_exp = c->d_boltz_fact = c->d_ltrans = c->d_freqs = c->d_logf = nullptr;
    if (!(c->n_lags > 2 && c->n_lags < 2 * kMaxTroughs && c->max_period <= 503 && c->n_bins >= 2 * c->trans_width && c->n_bins <= 384 &&
          c->trans_width >= 3 && (c->trans_width & 1))) {
        delete c;
        set_error("spev_pyin_create: (sr, fmin, fmax) outside what the kernels support");
        return SPEV_E_UNSUPPORTED;
    }
    // thresholds = linspace(0, 1, 101); beta_probs = diff(beta(2, 18).cdf(thresholds))
    std::vector<double> thr(c->n_thresholds + 1), cdf(c->n_thresholds + 1), bp(c->n_thresholds), bc(c->n_thresholds + 1, 0.0);
    const double step = 1.0 / c->n_thresholds;
    for (int i = 0; i <= c->n_thresholds; ++i) { thr[i] = i == c->n_thresholds ? 1.0 : i * step; cdf[i] = beta_cdf_int(thr[i], 2, 18); }
    for (int i = 0; i < c->n_thresholds; ++i) bp[i] = beta_probs_host ? beta_probs_host[i] : cdf[i + 1] - cdf[i];
    for (int i = 0; i < c->n_thresholds; ++i) bc[i + 1] = bc[i] + bp[i];
    // boltzmann.pmf(k, lambda=2, N) = (1 - e^-lambda) e^(-lambda k) / (1 - e^(-lambda N))
    const double lam = 2.0;
    std::vector<double> bexp(kMaxTroughs), bfact(kMaxTroughs + 1, 0.0);
    for (int k = 0; k < kMaxTroughs; ++k) bexp[k] = std::exp(-lam * k);
    for (int N = 1; N <= kMaxTroughs; ++N) bfact[N] = (1.0 - std::exp(-lam)) / (1.0 - std::exp(-lam * N));
    // transition = kron(transition_loop(2, 0.99), transition_local(n_bins, width, 'triangle')); log(. + tiny)
    const int W = c->trans_width, half = W / 2, nb = c->n_bins;
    c->n_classes = 2 * half + 1;
    std::vector<double> tri(W);
    for (int n = 0; n <= W / 2; ++n) tri[n] = tri[W - 1 - n] = 2.0 * (n + 1) / (W + 1.0);       // scipy.signal.triang(odd M)
    const double stay = 1.0 - 0.01, leave = (1.0 - stay) / 1.0;        // transition_loop(2, 1 - switch_prob)
    const double sw[2][2] = {{stay, leave}, {leave, stay}};
    std::vector<double> lt(static_cast<size_t>(4) * c->n_classes * W, kLogTiny64);
    for (int cls = 0; cls < c->n_classes; ++cls) {
        const int bprow = cls < half ? cls : (cls == half ? half : nb - half + (cls - half - 1));   // a representative row
        double rowsum = 0.0;
        for (int d = 0; d < W; ++d) { const int bcol = bprow + d - half; if (bcol >= 0 && bcol < nb) rowsum += tri[d]; }
        for (int vp = 0; vp < 2; ++vp)
            for (int v = 0; v < 2; ++v)
                for (int d = 0; d < W; ++d) {
                    // entry (from bp = bprow, to b = bprow + d' ) is stored at index (b - bp + half)
                    const int bcol = bprow + d - half;
                    if (bcol < 0 || bcol >= nb) continue;
                    const double tl = tri[d] / rowsum;
                    lt[((static_cast<size_t>(vp) * 2 + v) * c->n_classes + cls) * W + d] = std::log(sw[vp][v] * tl + kTiny64);
                }
    }
    c->h_ltrans = lt;
    c->h_beta = bp;
    c->h_freqs.resize(nb);
    for (int i = 0; i < nb; ++i) c->h_freqs[i] = fmin * std::pow(2.0, static_cast<double>(i) / (12.0 * c->bins_per_semitone));
    // device layout: (stay, switch) pairs; kron(switch, local) makes [0][0] == [1][1] and [0][1] == [1][0] bit for bit
    std::vector<double> ab(static_cast<size_t>(2) * c->n_classes * W);
    for (int i = 0; i < c->n_classes * W; ++i) {
        const size_t n1 = static_cast<size_t>(c->n_classes) * W;
        ab[2 * i] = lt[i];                 // [vp=0][v=0]
        ab[2 * i + 1] = lt[n1 + i];        // [vp=0][v=1]
        if (lt[3 * n1 + i] != lt[i] || lt[2 * n1 + i] != lt[n1 + i]) {
            delete c;
            set_error("spev_pyin_create: internal error, switch matrix not symmetric");
            return SPEV_E_INVALID;
        }
    }
    std::vector<double> logf(nb);
    for (int i = 0; i < nb; ++i) logf[i] = std::log(c->h_freqs[i] + 1e-8);
    int rc;
    if ((rc = upload(&c->d_thresholds, thr)) || (rc = upload(&c->d_beta_probs, bp)) || (rc = upload(&c->d_beta_cum, bc)) ||
        (rc = upload(&c->d_boltz_exp, bexp)) || (rc = upload(&c->d_boltz_fact, bfact)) || (rc = upload(&c->d_ltrans, ab)) ||
        (rc = upload(&c->d_freqs, c->h_freqs)) || (rc = upload(&c->d_logf, logf))) {
        spev_pyin_destroy(c);
        return rc;
    }
    *out = c;
    return SPEV_OK;
}

void spev_pyin_destroy(spev_pyin* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaFree(c->d_thresholds); cudaFree(c->d_beta_probs); cudaFree(c->d_beta_cum); cudaFree(c->d_boltz_exp);
    cudaFree(c->d_boltz_fact); cudaFree(c->d_ltrans); cudaFree(c->d_freqs); cudaFree(c->d_logf);
    delete c;
}

int spev_pyin_info(const spev_pyin* c, int* n_bins, int* min_period, int* max_period, int* n_lags) {
    SPEV_REQUIRE(c, SPEV_E_INVALID, "pyin ctx is null");
    if (n_bins) *n_bins = c->n_bins;
    if (min_period) *min_period = c->min_period;
    if (max_period) *max_period = c->max_period;
    if (n_lags) *n_lags = c->n_lags;
    return SPEV_OK;
}

int spev_pyin_host_tables(const spev_pyin* c, double* log_transition, double* freqs, double* beta_probs) {
    SPEV_REQUIRE(c, SPEV_E_INVALID, "pyin ctx is null");
    const int nb = c->n_bins, S = 2 * nb, W = c->trans_width, half = W / 2;
    if (log_transition) {                                  // dense [S, S], row = from-state
        for (int from = 0; from < S; ++from)
            for (int to = 0; to < S; ++to) {
                const int vp = from >= nb, bp = from - vp * nb, v = to >= nb, b = to - v * nb;
                double val = kLogTiny64;
                if (std::abs(b - bp) <= half) {
                    const int cls = bp < half ? bp : (bp >= nb - half ? half + 1 + (bp - (nb - half)) : half);
                    val = c->h_ltrans[((static_cast<size_t>(vp) * 2 + v) * c->n_classes + cls) * W + (b - bp + half)];
                }
                log_transition[static_cast<size_t>(from) * S + to] = val;
            }
    }
    if (freqs) std::copy(c->h_freqs.begin(), c->h_freqs.end(), freqs);
    if (beta_probs) std::copy(c->h_beta.begin(), c->h_beta.end(), beta_probs);
    return SPEV_OK;
}

int spev_pyin_cmnd(spev_pyin* c, const spev_batch* b, const float* samples, float* yin, void* stream) {
    SPEV_REQUIRE(c && b, SPEV_E_INVALID, "spev_pyin_cmnd: null ctx/batch");
    SPEV_CUDA(cudaSetDevice(c->device));
    if (b->n_frames == 0) return SPEV_OK;
    SPEV_REQUIRE(samples && yin && b->ftiles, SPEV_E_INVALID, "spev_pyin_cmnd: null buffer");
    const int64_t slots = static_cast<int64_t>(b->n_ftiles) * kTileFrames;
    const int grid = static_cast<int>(std::min<int64_t>(slots, 148 * 64));
    const int octets = ((c->max_period + 1 + 7) / 8 + 3) / 4 * 4;     // whole warps: 8 * octets threads
    const int threads = 8 * octets;
    {   // shared-partials kernel (default): one CTA per run of 16 frames
        const int L8 = 8 * octets, need = c->win_length + L8, zmax = (kCmndGroup - 1) * kHop + need, nplane = (zmax + 7) / 8 + 4;
        const size_t smem = sizeof(float) * (((zmax + 3) & ~3) + 4 * (2 * nplane + 4) + (2 * kCmndGroup + 6) * L8 +
                                             kCmndGroup * (need + 1) + 8);
        if (c->win_length == 1024 && c->frame_length == 2048 && smem <= 232448) {
            const int64_t groups = static_cast<int64_t>(b->n_ftiles) * ((kTileFrames + kCmndGroup - 1) / kCmndGroup);
            SPEV_CUDA(cudaFuncSetAttribute(k_yin_cmnd_shared, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
            k_yin_cmnd_shared<<<static_cast<int>(std::min<int64_t>(groups, 148 * 32)), kCmndThreads, smem, static_cast<cudaStream_t>(stream)>>>(
                view_of(b), samples, yin, c->frame_length, c->win_length, c->min_period, c->max_period, octets);
            SPEV_CUDA(cudaGetLastError());
            return SPEV_OK;
        }
    }
    k_yin_cmnd<<<grid, threads, sizeof(float) * (4096 + 16 + 2048 + 8 + kCmndSeg * threads + 32), static_cast<cudaStream_t>(stream)>>>(
        view_of(b), samples, yin, c->frame_length, c->win_length, c->min_period, c->max_period);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

int spev_pyin_observe(spev_pyin* c, const float* yin, int64_t n_frames, float* logobs, float* log_unvoiced,
                      float* voiced_prob, void* stream) {
    SPEV_REQUIRE(c, SPEV_E_INVALID, "spev_pyin_observe: null ctx");
    SPEV_CUDA(cudaSetDevice(c->device));
    SPEV_REQUIRE(n_frames >= 0, SPEV_E_INVALID, "spev_pyin_observe: n_frames < 0");
    if (n_frames == 0) return SPEV_OK;
    SPEV_REQUIRE(yin && logobs && log_unvoiced && voiced_prob, SPEV_E_INVALID, "spev_pyin_observe: null buffer");
    ObsParams p{c->n_lags, c->min_period, c->n_thresholds, c->n_bins, c->bins_per_semitone, c->sr, c->fmin,
                c->no_trough_prob, c->d_thresholds, c->d_beta_probs, c->d_beta_cum, c->d_boltz_exp, c->d_boltz_fact};
    const int grid = static_cast<int>(std::min<int64_t>(n_frames, 148 * 64));
    k_pyin_observe<<<grid, kObsThreads, 0, static_cast<cudaStream_t>(stream)>>>(yin, n_frames, p, logobs, log_unvoiced, voiced_prob);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

size_t spev_pyin_decode_workspace_bytes(const spev_pyin* c, int64_t n_frames) {
    if (!c || n_frames < 0) return 0;
    return static_cast<size_t>(n_frames) * 2 * c->n_bins * sizeof(unsigned short) + 512;
}

int spev_pyin_decode(spev_pyin* c, const float* logobs, const float* log_unvoiced, const int64_t* frame_off, int n_items,
                     int64_t n_frames, int32_t* states, float* f0, uint8_t* voiced_flag, void* workspace,
                     size_t workspace_bytes, void* stream) {
    SPEV_REQUIRE(c, SPEV_E_INVALID, "spev_pyin_decode: null ctx");
    SPEV_CUDA(cudaSetDevice(c->device));
    SPEV_REQUIRE(n_items >= 0 && n_frames >= 0, SPEV_E_INVALID, "spev_pyin_decode: negative sizes");
    if (n_items == 0 || n_frames == 0) return SPEV_OK;
    SPEV_REQUIRE(logobs && log_unvoiced && frame_off && states, SPEV_E_INVALID, "spev_pyin_decode: null buffer");
    SPEV_REQUIRE(workspace && workspace_bytes >= spev_pyin_decode_workspace_bytes(c, n_frames), SPEV_E_WORKSPACE,
                 "spev_pyin_decode: workspace too small");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    unsigned* counter = reinterpret_cast<unsigned*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    unsigned short* ptr = reinterpret_cast<unsigned short*>(counter + 64);
    SPEV_REQUIRE(c->n_bins <= kVitThreads, SPEV_E_UNSUPPORTED, "spev_pyin_decode: too many pitch bins");
    const size_t tab_bytes = sizeof(double2) * static_cast<size_t>(c->n_classes) * c->trans_width;
    const bool tab_smem = tab_bytes <= 96 * 1024;              // two CTAs per SM
    VitParams p{c->n_bins, c->trans_width, c->n_classes, reinterpret_cast<const double2*>(c->d_ltrans)};
    const size_t smem = sizeof(double2) * static_cast<size_t>(2) * c->n_bins + (tab_smem ? tab_bytes : 0);
    auto kern = tab_smem ? k_pyin_viterbi<true> : k_pyin_viterbi<false>;
    SPEV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    SPEV_CUDA(cudaMemsetAsync(counter, 0, sizeof(unsigned), st));
    const int grid = std::min(n_items, 148 * SPEV_VIT_CTAS);
    kern<<<grid, kVitThreads, smem, st>>>(logobs, log_unvoiced, frame_off, n_items, p, ptr, states, counter);
    SPEV_CUDA(cudaGetLastError());
    if (f0 || voiced_flag) {
        const int g2 = static_cast<int>(std::min<int64_t>((n_frames + 255) / 256, 148 * 8));
        k_pyin_finish<<<g2, 256, 0, st>>>(states, n_frames, c->n_bins, c->d_freqs, f0, voiced_flag);
        SPEV_CUDA(cudaGetLastError());
    }
    return SPEV_OK;
}

int spev_pitch_pool(const spev_pyin* c, const int32_t* states, const int64_t* frame_off, const int64_t* durs,
                    const int64_t* phone_off, int n_items, double p_mean, double p_std, float lo, float hi, float rough_hi,
                    float* pitch, float* rough, void* stream) {
    SPEV_REQUIRE(c, SPEV_E_INVALID, "spev_pitch_pool: null ctx");
    SPEV_CUDA(cudaSetDevice(c->device));
    SPEV_REQUIRE(n_items >= 0, SPEV_E_INVALID, "spev_pitch_pool: n_items < 0");
    if (n_items == 0) return SPEV_OK;
    SPEV_REQUIRE(states && frame_off && durs && phone_off && pitch && rough, SPEV_E_INVALID, "spev_pitch_pool: null buffer");
    SPEV_REQUIRE(p_std != 0.0, SPEV_E_INVALID, "spev_pitch_pool: p_std == 0");
    const int wpb = 4;
    const int grid = std::min((n_items + wpb - 1) / wpb, 148 * 16);
    k_pitch_pool<<<grid, wpb * 32, 0, static_cast<cudaStream_t>(stream)>>>(
        states, frame_off, reinterpret_cast<const long long*>(durs), phone_off, n_items, c->n_bins, c->d_logf, p_mean, p_std,
        lo, hi, rough_hi, pitch, rough);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

}  // extern "C"

