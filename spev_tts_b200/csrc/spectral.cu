// spectral.cu -- STFT / mel / ISTFT / Griffin-Lim kernels for sm_100a.
//
// K1 k_stft_mel   : frames -> Hann -> rFFT-1024 (two frames per warp transform) -> |X|^2 ->
//                   banded Slaney-mel FFMA epilogue -> log/clamp -> [F, n_mels]
//                   (or, MODE 1, the raw power spectrum [F, 520] for the tcgen05 GEMM path).
//                   Replaces /root/reference/spev_real_metrics.py:363-367.
// K4 k_istft      : two Hermitian spectra per warp -> irFFT-1024 -> Hann -> shared memory;
//                   gather overlap-add (each output sample owner sums its <= 4 frames in
//                   ascending frame order, no atomics) fused with window-sum-square
//                   normalisation.            Replaces librosa.istft under :730-733.
//                   Chunk tiles carry each item's output bounds [lo, hi) (librosa's istft(length=)):
//                   every sample of [lo, hi) is written, nothing outside it.
// K5 k_stft_phase_w : STFT of the rebuilt signal fused with Griffin-Lim's momentum / phase
//                   normalisation update, one frame pair per warp.  Replaces librosa.stft + the angle
//                   update lines of librosa.griffinlim under :730-733.
// K5f k_gl_fused  : the Griffin-Lim ITERATION as the driver runs it (round 2): STFT + phase update + inverse transform of
//                   the new spectra in registers; leaves one overlap-add segment per frame pair.  K4p k_ola_pairs sums the
//                   segments into y.  (K4 / K5 above stay the stand-alone spev_istft / spev_stft / spev_gl_phase_update.)
// K3 k_mel_to_mag : S = sqrt(max(pinv . exp(logmel), 0)) (FFMA version; the tcgen05 version
//                   lives in gemm_tc.cu).     Replaces librosa mel_to_stft under :730.
//
// All FFT kernels are persistent (grid = #SMs, one 16-warp CTA per SM).  K1 and K4 go round-robin
// over host-built 48-byte tile descriptors, and nothing on their per-tile critical path waits on
// global memory: tile descriptors travel through a 4-slot cp.async ring three tiles ahead, and
// the samples of tile i+1 are cp.async-staged into the second half of a double buffer while
// tile i is transformed.  K5 and K5f hand out frame pairs to warps instead (see k_stft_phase_w).
//
// Shared-memory plan per CTA (K1 / K4):
//   s_tw    float2[32*32]   inter-stage twiddles                       8,192 B
//   s_win   float [1024]    periodic Hann                              4,096 B
//   s_ring  spev_tile[4]    descriptor ring                              192 B
//   s_stage float [2][8960] double-buffered tile samples (K1)         71,680 B
//   s_x     16 x 2114 words warp-private transpose tiles; reused for
//                           |X|^2 (K1) / windowed frames (K4)        135,296 B
//   bands   CSR form of the mel basis (K1)                            ~5,000 B
#include <algorithm>
#include "spev_internal.cuh"
#include "tile_pipe.cuh"

namespace spev {

// s_win holds win_scale * Hann: 0.5 for the forward kernels (folds the 1/2 of the Hermitian split
// into the window -- exact, a power of two), 1 for the inverse kernel.
__device__ __forceinline__ void load_tables(float2* s_tw, float* s_win, const float2* __restrict__ g_tw,
                                            const float* __restrict__ g_win, float win_scale) {
    for (int i = threadIdx.x; i < 1024; i += blockDim.x) {
        s_tw[i] = g_tw[i];
        s_win[i] = win_scale * g_win[i];
    }
}

// Asynchronously stage samples x[src0 .. src0+count) (zero outside [lo, hi)) into shared memory.
__device__ __forceinline__ void stage_async(float* s_stage, const float* __restrict__ x,
                                            const spev_tile& d) {
    const int count = (d.n - 1) * kHop + kNfft;
    const int64_t first = d.src0;
    // tile-local valid range [i_lo, i_hi): 32-bit from here on
    const int i_lo = static_cast<int>(max(static_cast<int64_t>(0), d.lo - first));
    const int i_hi = static_cast<int>(min(static_cast<int64_t>(count), d.hi - first));
    const float* xs = x + first;
    const bool vec_ok = ((reinterpret_cast<uintptr_t>(x) & 15) == 0) && ((d.lo & 3) == 0);
    if (vec_ok) {   // lo % 4 == 0 and first == lo (mod 4): a float4 never straddles `lo`
        // [0, a4) lies before the item (zero fill), [a4, b4) are whole 16-byte chunks inside it -- the only
        // non-empty range for interior tiles, copied by a loop without any bounds arithmetic --, [b4, count)
        // holds the chunk that straddles `hi` and the zero fill after it.
        const int a4 = min(count, i_lo), b4 = max(a4, min(count, i_hi) & ~3);
        const int step = blockDim.x * 4;
        for (int i = threadIdx.x * 4; i < a4; i += step) cp_async16(s_stage + i, x, 0);
        for (int i = a4 + threadIdx.x * 4; i < b4; i += step) cp_async16(s_stage + i, xs + i, 16);
        for (int i = b4 + threadIdx.x * 4; i < count; i += step) {
            const int nb = max(0, min(16, (i_hi - i) * 4));
            cp_async16(s_stage + i, nb > 0 ? xs + i : x, nb);
        }
    } else {
        for (int i = threadIdx.x; i < count; i += blockDim.x) {
            const bool ok = i >= i_lo && i < i_hi;
            cp_async4(s_stage + i, ok ? xs + i : x, ok ? 4 : 0);
        }
    }
}

// Load the two windowed frames a (real part) and b (imaginary part) of this warp from the
// staged samples: v[j] = win[32j+lane] * (stage[256a + 32j + lane], stage[256b + 32j + lane]).
// Frame b of an odd tile tail does not exist: its slot must be exactly zero (anything else would
// leak rounding error into frame a through the packed transform), hence the warp-uniform branch.
__device__ __forceinline__ void load_frame_pair(float2 (&v)[32], const float* s_stage,
                                                const float* s_win, int fa, bool b_valid, int lane) {
    const float* pa = s_stage + fa * kHop + lane;
    if (b_valid) {
        // frame b = frame a shifted by one hop (8 rows of 32): 40 loads serve both frames
        float x[40];
        static_for<0, 40>([&](auto jc) {
            constexpr int j = decltype(jc)::value;
            x[j] = pa[32 * j];
        });
        static_for<0, 32>([&](auto jc) {
            constexpr int j = decltype(jc)::value;
            const float w = s_win[32 * j + lane];
            v[j] = make_float2(w * x[j], w * x[j + 8]);
        });
    } else {
        static_for<0, 32>([&](auto jc) {
            constexpr int j = decltype(jc)::value;
            v[j] = make_float2(s_win[32 * j + lane] * pa[32 * j], 0.f);
        });
    }
}

// ---------------------------------------------------------------------------------------
// Mel phase of the fused log-mel kernel: lane <-> frame (pf = the lane's |X|^2 row, conflict-free LDS.128),
// warp <-> its NB bands.  Per float4 group: one broadcast LDS.128 of weights, one LDS.128 of |X|^2, four FFMA --
// no index loads, no per-group branch (a band is a run of consecutive bins); the NB results stay in registers
// until all bands are done, so nothing orders the loads behind a store and they pipeline freely.
// NB == 0: run-time band count (n_mels > 128).
// ---------------------------------------------------------------------------------------
template <int NB>
__device__ __forceinline__ void mel_bands(const float* __restrict__ pf, const float4* __restrict__ s_gw,
                                          const int4* __restrict__ hdr, int nb_rt, float* __restrict__ s_row,
                                          int log_mode, float floor_v, float lo, float hi) {
    auto band = [&](const int4 h) {
        const float4* wv = s_gw + h.x;
        const float* px = pf + h.y;
        float acc0 = 0.f, acc1 = 0.f;
#pragma unroll 2
        for (int g = 0; g < h.z; ++g) {
            const float4 w = wv[g];
            const float4 x = *reinterpret_cast<const float4*>(px + 4 * g);
            acc0 = fmaf(w.x, x.x, acc0);
            acc1 = fmaf(w.y, x.y, acc1);
            acc0 = fmaf(w.z, x.z, acc0);
            acc1 = fmaf(w.w, x.w, acc1);
        }
        float acc = acc0 + acc1;
        // __logf: <= 3 ulp (2^-21.4 abs in [0.5,2]) -- far inside the 1e-4 tolerance
        if (log_mode) acc = fminf(fmaxf(__logf(fmaxf(acc, floor_v)), lo), hi);
        return acc;
    };
    if constexpr (NB > 0) {
        float r[NB];
        int mel[NB];
        static_for<0, NB>([&](auto bc) {
            constexpr int b = decltype(bc)::value;
            const int4 h = hdr[b];
            r[b] = band(h);
            mel[b] = h.w;
        });
        static_for<0, NB>([&](auto bc) {
            constexpr int b = decltype(bc)::value;
            if (mel[b] >= 0) s_row[mel[b]] = r[b];
        });
    } else {
        for (int b = 0; b < nb_rt; ++b) {
            const int4 h = hdr[b];
            const float r = band(h);
            if (h.w >= 0) s_row[h.w] = r;
        }
    }
}

// ---------------------------------------------------------------------------------------
// K1: fused STFT -> power -> mel -> log
// ---------------------------------------------------------------------------------------
template <int MODE, int NB>   // MODE 0: mel epilogue (NB bands per warp, 0 = run time), 1: power-spectrum output
__global__ void __launch_bounds__(kThreads, 1)
k_stft_mel(BatchView bv, const float* __restrict__ samples, float* __restrict__ out,
           const float2* __restrict__ g_tw, const float* __restrict__ g_win, MelProgram mb,
           int log_mode, float floor_v, float lo, float hi) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* s_tw = reinterpret_cast<float2*>(smem_raw);
    float* s_win = reinterpret_cast<float*>(s_tw + 1024);
    spev_tile* s_ring = reinterpret_cast<spev_tile*>(s_win + 1024);
    float* s_stage = reinterpret_cast<float*>(s_ring + kRing);
    float* s_x = s_stage + 2 * kStageSamples;
    float4* s_gw = reinterpret_cast<float4*>(s_x + kWarps * kWarpRegionWords);   // [n_groups], 16-B aligned
    int4* s_hdr = reinterpret_cast<int4*>(s_gw + mb.n_groups);                   // [16*nb]

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    load_tables(s_tw, s_win, g_tw, g_win, 0.5f);
    if (MODE == 0) {
        for (int i = threadIdx.x; i < mb.n_groups; i += blockDim.x) s_gw[i] = mb.gw[i];
        for (int i = threadIdx.x; i < kWarps * mb.nb; i += blockDim.x) s_hdr[i] = mb.hdr[i];
    }
    float* xw = s_x + warp * kWarpRegionWords;
    const int n_mels = mb.n_mels;
    const int out_pitch = n_mels + 1;
    // output copy mapping: thread <-> (frame residue, mel bin), fixed for the whole kernel
    const int rows_per_pass = kThreads / n_mels;
    const int cp_m = threadIdx.x % n_mels, cp_f0 = threadIdx.x / n_mels;

    const int stride = gridDim.x;
    const int my_n = ring_prologue(s_ring, bv.ftiles, bv.n_ftiles);
    if (my_n > 0) stage_async(s_stage, samples, s_ring[0]);
    cp_async_commit();

    for (int i = 0; i < my_n; ++i) {
        cp_async_wait_all();
        __syncthreads();   // B1: tile i staged + visible; previous tile fully consumed
        const int nf = s_ring[i & 3].n;
        const int64_t row0 = s_ring[i & 3].row0;
        if (i + 1 < my_n) stage_async(s_stage + ((i + 1) & 1) * kStageSamples, samples, s_ring[(i + 1) & 3]);
        if (i + 3 < my_n) fetch_desc(s_ring + ((i + 3) & 3), bv.ftiles + blockIdx.x + (i + 3) * stride);
        cp_async_commit();
        float* stage = s_stage + (i & 1) * kStageSamples;

        const int fa = 2 * warp;
        if (fa < nf) {
            const bool b_valid = fa + 1 < nf;
            float2 v[32];
            load_frame_pair(v, stage, s_win, fa, b_valid, lane);
            warp_fft1024<-1>(v, reinterpret_cast<float2*>(xw), s_tw, lane);
            float2 p[16];
            fetch_mirror(v, p, lane);
            __syncwarp();   // transpose tile is dead; reuse it for |X|^2
            // lane 0: bin 512 (the window carries a factor 1/2: X[512] = 2 * Z'[512])
            const float pa512 = 4.f * v[16].x * v[16].x, pb512 = 4.f * v[16].y * v[16].y;
            if (MODE == 0) {
                static_for<0, 16>([&](auto kc) {
                    constexpr int k2 = decltype(kc)::value;
                    float2 xa, xb;
                    split_pair_prescaled(v[k2], p[k2], xa, xb);
                    xw[lane + 32 * k2] = fmaf(xa.x, xa.x, xa.y * xa.y);
                    xw[kPSlot + lane + 32 * k2] = fmaf(xb.x, xb.x, xb.y * xb.y);
                });
                if (lane < 4) {   // bin 512 + three zero words so that padded float4 band reads stay clean
                    xw[512 + lane] = lane == 0 ? pa512 : 0.f;
                    xw[kPSlot + 512 + lane] = lane == 0 ? pb512 : 0.f;
                }
            } else {
                float* oa = out + (row0 + fa) * kSpecLd;
                float* ob = oa + kSpecLd;
                static_for<0, 16>([&](auto kc) {
                    constexpr int k2 = decltype(kc)::value;
                    float2 xa, xb;
                    split_pair_prescaled(v[k2], p[k2], xa, xb);
                    oa[lane + 32 * k2] = fmaf(xa.x, xa.x, xa.y * xa.y);
                    if (b_valid) ob[lane + 32 * k2] = fmaf(xb.x, xb.x, xb.y * xb.y);
                });
                if (lane < kSpecLd - 512) {   // bin 512 + zero pad columns 513..519
                    oa[512 + lane] = lane == 0 ? pa512 : 0.f;
                    if (b_valid) ob[512 + lane] = lane == 0 ? pb512 : 0.f;
                }
            }
        }
        if (MODE == 0) {
            __syncthreads();   // B2: all |X|^2 written; this tile's samples no longer read
            // mel phase: lane <-> frame (conflict-free: bank = frame + bin), warp <-> band set
            // mel phase: lane <-> frame (conflict-free: bank group = frame), warp <-> band program.
            // Results are staged in shared memory (the consumed half of the sample double buffer) and
            // copied out as contiguous rows; storing 4-byte values straight from this loop was
            // measured slower (650 vs 702 M frames/s: 32 sectors per store instruction).
            float* s_out = stage;
            // lanes >= nf run on stale slots; their rows are never copied out (no divergence)
            mel_bands<NB>(s_x + (lane >> 1) * kWarpRegionWords + (lane & 1) * kPSlot, s_gw, s_hdr + warp * mb.nb, mb.nb,
                          s_out + lane * out_pitch, log_mode, floor_v, lo, hi);
            __syncthreads();   // B3
            float* o = out + row0 * n_mels;
            if (cp_f0 < rows_per_pass)
                for (int f = cp_f0; f < nf; f += rows_per_pass) o[f * n_mels + cp_m] = s_out[f * out_pitch + cp_m];
        }
    }
}

// ---------------------------------------------------------------------------------------
// Griffin-Lim phase update of one bin: a = reb - alpha * tprev (unless has_prev == 0), S * a / (|a| + tiny)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float2 phase_of(float2 reb, float s, float2 tp, float alpha, int has_prev) {
    float2 a = reb;
    if (has_prev) {
        a.x = a.x - alpha * tp.x;
        a.y = a.y - alpha * tp.y;
    }
    const float den = sqrtf(fmaf(a.x, a.x, a.y * a.y)) + kTiny;
    const float r = 1.0f / den;   // numpy complex/real division multiplies by the reciprocal
    return make_float2(a.x * r * s, a.y * r * s);
}

// ---------------------------------------------------------------------------------------
// K5w: warp-independent STFT (+ Griffin-Lim phase update)
//
// The phase update has no cross-warp data dependence, so here every warp is its own worker:
// it takes (tile, slot) pairs one at a time, cp.async-stages the 1280 samples of its NEXT pair
// into a warp-private buffer as soon as the current pair's samples are in registers (the copy has
// the whole transform to land), and never meets a CTA barrier.  Warps drift out of phase, so the
// FFTs of some overlap the L2/HBM epilogues of others instead of the whole SM alternating between
// "compute only" and "memory only".
// ---------------------------------------------------------------------------------------
struct PairInfo {
    int64_t row;      // global row of frame a
    int valid;        // 0: no such pair
    int b_valid;
};

__device__ __forceinline__ PairInfo stage_pair(float* region, const float* __restrict__ x, const spev_tile* __restrict__ tiles,
                                               int64_t p, int64_t n_pairs, int lane) {
    PairInfo pi{0, 0, 0};
    if (p >= n_pairs) return pi;
    const spev_tile* d = tiles + (p >> 4);
    const int fa = 2 * static_cast<int>(p & 15);
    const int n = __ldg(&d->n);
    if (fa >= n) return pi;
    const int64_t src0 = __ldg(&d->src0), lo = __ldg(&d->lo), hi = __ldg(&d->hi);
    pi.row = __ldg(&d->row0) + fa;
    pi.valid = 1;
    pi.b_valid = fa + 1 < n;
    const int count = kNfft + kHop;                       // samples of frames a and a+1
    const int64_t first = src0 + static_cast<int64_t>(fa) * kHop;
    const int i_lo = static_cast<int>(max(static_cast<int64_t>(0), lo - first));
    const int i_hi = static_cast<int>(min(static_cast<int64_t>(count), hi - first));
    const float* xs = x + first;
    if (((reinterpret_cast<uintptr_t>(x) & 15) == 0) && ((lo & 3) == 0)) {
#pragma unroll
        for (int j = 0; j < count / 128; ++j) {
            const int i = lane * 4 + 128 * j;
            int nb = i >= i_lo ? (i_hi - i) * 4 : 0;
            nb = max(0, min(16, nb));
            cp_async16(region + i, nb > 0 ? xs + i : x, nb);
        }
    } else {
        for (int i = lane; i < count; i += 32) {
            const bool ok = i >= i_lo && i < i_hi;
            cp_async4(region + i, ok ? xs + i : x, ok ? 4 : 0);
        }
    }
    return pi;
}

// Work distribution: warp w of CTA c takes pairs w + 16 c, then strides by 16 * grid.
// STAGE_T (phase update only): the pair's `tprev` rows are pulled into the warp's transpose tile by ONE bulk
// asynchronous copy (cp.async.bulk, 8,272 B) as soon as the exchange has been read back; it lands during the second
// 32-point DFT, so the epilogue reads them from shared memory instead of waiting on 32 global loads per lane
// (ncu before: long_scoreboard 2.5 warps per issue cycle on exactly those loads).
constexpr int kWsRegionWords = kXWords + kNfft + kHop;   // transpose tile + 1280 staged samples of the NEXT pair

template <int MODE, bool STAGE_T>   // MODE 0: plain STFT into `ang`; 1: Griffin-Lim phase update
__global__ void __launch_bounds__(kThreads, 1)
k_stft_phase_w(BatchView bv, const float* __restrict__ y, const float* __restrict__ S, int64_t ld_s,
               float2* __restrict__ ang, float2* tprev, int64_t ld, float alpha, int has_prev,
               const float2* __restrict__ g_tw, const float* __restrict__ g_win) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* s_tw = reinterpret_cast<float2*>(smem_raw);
    float* s_win = reinterpret_cast<float*>(s_tw + 1024);
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_win + 1024);        // one mbarrier per warp
    float* s_x = reinterpret_cast<float*>(s_bar + kWarps);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    pdl_launch_dependents();
    load_tables(s_tw, s_win, g_tw, g_win, 0.5f);
    if (STAGE_T && threadIdx.x < kWarps) bar_init(s_bar + threadIdx.x, 1);
    if (STAGE_T && threadIdx.x == 0) asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    __syncthreads();                                     // the only CTA-wide barrier
    float* tile = s_x + warp * kWsRegionWords;           // exchange tile, then the staged tprev rows
    float* xs = tile + kXWords;                          // samples of the pair being loaded / staged next
    float2* xb = reinterpret_cast<float2*>(tile);
    uint64_t* tbar = s_bar + warp;
    unsigned tphase = 0;

    const int64_t n_pairs = static_cast<int64_t>(bv.n_ftiles) * kWarps;
    const int64_t stride = static_cast<int64_t>(gridDim.x) * kWarps;
    int64_t p_next = static_cast<int64_t>(blockIdx.x) * kWarps + warp;
    // stage the samples of this warp's next pair that has frames (slots past a partial tile's end have none)
    auto stage_next = [&]() -> PairInfo {
        PairInfo pi{0, 0, 0};
        for (;;) {
            const int64_t p = p_next;
            p_next += stride;
            if (p >= n_pairs) return pi;
            pi = stage_pair(xs, y, bv.ftiles, p, n_pairs, lane);
            if (pi.valid) return pi;
        }
    };
    pdl_wait();                                          // y / ang / tprev come from the previous kernel
    PairInfo cur = stage_next();
    cp_async_commit();

    while (cur.valid) {
        cp_async_wait_all();
        __syncwarp();
        float2 v[32];
        load_frame_pair(v, xs, s_win, 0, cur.b_valid != 0, lane);
        __syncwarp();                                    // staged samples consumed
        // ---- stage the next pair's samples now: they have this whole pair's time to arrive ----
        const PairInfo nxt = stage_next();
        cp_async_commit();
        const bool b_valid = cur.b_valid != 0;
        const int64_t ra = cur.row * ld, rb = ra + ld;
        const float* sa = S + cur.row * ld_s;
        const float* sb = sa + ld_s;
        if (MODE == 1) {                                 // pull this pair's S rows (and tprev, unless staged) into L2
            const int rows = b_valid ? 2 : 1;
            warp_prefetch_l2(sa, static_cast<int>((rows - 1) * ld_s + kBins) * 4, lane);
            if (!STAGE_T && has_prev) warp_prefetch_l2(tprev + ra, static_cast<int>((rows - 1) * ld + kBins) * 8, lane);
        }
        // ---- first half of the transform: 32-point DFTs, inter-stage twiddles, transpose ----
        dft32<-1>(v);
        static_for<1, 32>([&](auto k1c) {
            constexpr int k1 = decltype(k1c)::value;
            v[k1] = cmul(v[k1], s_tw[k1 * 32 + lane]);
        });
        static_for<0, 32>([&](auto k1c) {
            constexpr int k1 = decltype(k1c)::value;
            xb[k1 * kXPitch + lane] = v[k1];
        });
        __syncwarp();
        static_for<0, 32>([&](auto n2c) {
            constexpr int n2 = decltype(n2c)::value;
            v[n2] = xb[lane * kXPitch + n2];
        });
        __syncwarp();                                    // tile read back: free for the tprev rows
        const bool staged = STAGE_T && MODE == 1 && has_prev;
        if (staged) {
            const uint32_t bytes = b_valid ? static_cast<uint32_t>(ld * 8 + (kBins + 1) * 8) : static_cast<uint32_t>((kBins + 1) * 8);
            if (lane == 0) {
                fence_proxy_async();
                bar_expect_tx(tbar, bytes);
                bulk_g2s(tile, tprev + ra, bytes, tbar);
            }
        }
        dft32<-1>(v);
        float2 pm[16];
        fetch_mirror(v, pm, lane);
        const float2* tsm = reinterpret_cast<const float2*>(tile);   // staged rows: a at [0, 514), b at [ld, ld + 514)
        if (staged) { bar_wait(tbar, tphase); tphase ^= 1; }
        static_for<0, 4>([&](auto gc) {
            constexpr int g = decltype(gc)::value;
            float2 tpa[4], tpb[4];
            float s_a[4], s_b[4];
            if (MODE == 1) {
                static_for<0, 4>([&](auto qc) {
                    constexpr int q = decltype(qc)::value;
                    const int k = lane + 32 * (4 * g + q);
                    s_a[q] = sa[k];
                    s_b[q] = b_valid ? sb[k] : 0.f;
                    if (staged) {
                        tpa[q] = tsm[k];
                        tpb[q] = b_valid ? tsm[ld + k] : make_float2(0.f, 0.f);
                    } else {
                        tpa[q] = has_prev ? tprev[ra + k] : make_float2(0.f, 0.f);
                        tpb[q] = (has_prev && b_valid) ? tprev[rb + k] : make_float2(0.f, 0.f);
                    }
                });
            }
            static_for<0, 4>([&](auto qc) {
                constexpr int q = decltype(qc)::value;
                constexpr int k2 = 4 * g + q;
                const int k = lane + 32 * k2;
                float2 xa, xbv;
                split_pair_prescaled(v[k2], pm[k2], xa, xbv);
                if (MODE == 0) {
                    ang[ra + k] = xa;
                    if (b_valid) ang[rb + k] = xbv;
                } else {
                    ang[ra + k] = phase_of(xa, s_a[q], tpa[q], alpha, has_prev);
                    tprev[ra + k] = xa;
                    if (b_valid) {
                        ang[rb + k] = phase_of(xbv, s_b[q], tpb[q], alpha, has_prev);
                        tprev[rb + k] = xbv;
                    }
                }
            });
        });
        if (lane == 0) {
            // the window carries a factor 1/2: X[512] = 2 * Z'[512]
            const float2 xa = make_float2(2.f * v[16].x, 0.f), xbv = make_float2(2.f * v[16].y, 0.f);
            if (MODE == 0) {
                ang[ra + 512] = xa;
                if (b_valid) ang[rb + 512] = xbv;
            } else {
                const float2 z = make_float2(0.f, 0.f);
                const float2 ta = !has_prev ? z : (staged ? tsm[512] : tprev[ra + 512]);
                ang[ra + 512] = phase_of(xa, sa[512], ta, alpha, has_prev);
                tprev[ra + 512] = xa;
                if (b_valid) {
                    const float2 tb = !has_prev ? z : (staged ? tsm[ld + 512] : tprev[rb + 512]);
                    ang[rb + 512] = phase_of(xbv, sb[512], tb, alpha, has_prev);
                    tprev[rb + 512] = xbv;
                }
            }
        }
        __syncwarp();                                    // staged rows consumed: the tile is free for the next exchange
        cur = nxt;
    }
}

// ---------------------------------------------------------------------------------------
// K5f: the fused Griffin-Lim iteration (default since r02): STFT of the rebuilt signal, momentum / phase update, and
// the INVERSE transform of the new spectra without leaving the registers; what goes back to HBM is the pair's
// 1280-sample overlap-add segment (k_ola_pairs finishes the overlap-add) and the rebuilt spectra for the momentum term.
//
// Same staging as k_stft_phase_w (warp-independent pairs, cp.async samples one pair ahead, bulk-staged tprev rows),
// but the body is written ONCE and run twice per pair: pass 0 transforms the samples, pass 1 the new spectra.  The
// inverse transform is the forward one on swapped components (swap(z) = i conj(z): ifft(V) = swap(fft(swap(V)))), so
// both passes -- and, inside a pass, both 32-point stages -- execute the same instructions.  A straight-line body (four
// inlined 32-point DFTs, ~75 KB of code) was measured: it lost 1.3 warps per issue cycle to instruction fetch (ncu
// `no_instruction`) because its 16 drifting warps walk the whole body at different places; this body is less than
// half of that.
// Work distribution: with `counter` the warps draw (tile, slot) pairs dynamically (draw_ticket) -- worth it once a
// warp has many pairs, see launch_stft_phase --, else they stride statically like k_stft_phase_w.
// ---------------------------------------------------------------------------------------
// phase_of with the |a| normalisation by MUFU.RSQ (2 ulp) instead of IEEE sqrt + divide
__device__ __forceinline__ float2 phase_of_rsqrt(float2 reb, float s, float2 tp, float alpha, int has_prev) {
    float2 a = reb;
    if (has_prev) {
        a.x = a.x - alpha * tp.x;
        a.y = a.y - alpha * tp.y;
    }
    // 1 / (|a| + tiny) == rsqrt(|a|^2) wherever |a|^2 is a normal number; the clamp keeps a == 0 at 0 * finite
    const float n2 = fmaxf(fmaf(a.x, a.x, a.y * a.y), 1e-36f);
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(n2));
    r *= s;
    return make_float2(a.x * r, a.y * r);
}

template <bool STAGE_T>
__global__ void __launch_bounds__(kThreads, 1)
k_gl_fused(BatchView bv, const float* __restrict__ y, const float* __restrict__ S, int64_t ld_s,
           float* __restrict__ seg_base, float2* tprev, int64_t ld, float alpha, int has_prev,
           const float2* __restrict__ g_tw, const float* __restrict__ g_win, unsigned* counter, unsigned base) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* s_tw = reinterpret_cast<float2*>(smem_raw);
    float* s_win = reinterpret_cast<float*>(s_tw + 1024);
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_win + 1024);        // two mbarriers per warp: tprev rows, S rows
    float* s_x = reinterpret_cast<float*>(s_bar + 2 * kWarps);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    pdl_launch_dependents();
    load_tables(s_tw, s_win, g_tw, g_win, 0.5f);
    if (STAGE_T && threadIdx.x < 2 * kWarps) bar_init(s_bar + threadIdx.x, 1);
    if (STAGE_T && threadIdx.x == 0) asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    __syncthreads();                                     // the only CTA-wide barrier
    float* tile = s_x + warp * kWsRegionWords;           // exchange tile, then the staged tprev rows
    float* xs = tile + kXWords;                          // samples of the pair being loaded / staged next
    float2* xb = reinterpret_cast<float2*>(tile);
    uint64_t* tbar = s_bar + warp;
    uint64_t* sbar = s_bar + kWarps + warp;
    unsigned tphase = 0, sphase = 0;
    const int pl = (32 - lane) & 31;
    // tprev streams through (read once, rewritten, next use a whole iteration away); S and the segments are re-used soon.
    // The broadcast from lane 0 keeps the policies in uniform registers: without it ptxas moves them to per-thread
    // registers and converts them back before each of the ~50 hinted stores (measured 1 % slower at cfg3).
    const uint64_t pol_stream = __shfl_sync(0xffffffffu, l2_policy_evict_first(), 0);
    const uint64_t pol_keep = __shfl_sync(0xffffffffu, l2_policy_evict_last(), 0);

    const int64_t n_pairs = static_cast<int64_t>(bv.n_ftiles) * kWarps;
    const int64_t stride = static_cast<int64_t>(gridDim.x) * kWarps;
    int64_t p_static = static_cast<int64_t>(blockIdx.x) * kWarps + warp;
    bool drained = false;
    unsigned pend = 0;
    auto draw_ahead = [&]() { if (lane == 0) pend = draw_ticket(counter, base); };
    auto next_pair = [&]() -> int64_t {
        if (counter == nullptr) { const int64_t p = p_static; p_static += stride; return p; }
        if (drained) return n_pairs;
        const unsigned t = __shfl_sync(0xffffffffu, pend, 0);
        if (t >= static_cast<unsigned>(n_pairs)) { drained = true; return n_pairs; }
        draw_ahead();
        return static_cast<int64_t>(t);
    };
    auto stage_next = [&]() -> PairInfo {
        PairInfo pi{0, 0, 0};
        for (;;) {
            const int64_t p = next_pair();
            if (p >= n_pairs) return pi;
            pi = stage_pair(xs, y, bv.ftiles, p, n_pairs, lane);
            if (pi.valid) return pi;
        }
    };
    pdl_wait();                                          // y / tprev come from the previous kernels
    // Tickets may only be drawn once every earlier launch of this kernel has finished drawing: with programmatic
    // dependent launch the prologue above can run while the launch before the previous kernel is still at work, and
    // its tickets would interleave with ours.  griddepcontrol.wait returns when the whole chain behind us is complete.
    if (counter != nullptr) draw_ahead();
    PairInfo cur = stage_next();
    cp_async_commit();

    while (cur.valid) {
        cp_async_wait_all();
        __syncwarp();
        const bool b_valid = cur.b_valid != 0;
        float2 v[32];
        load_frame_pair(v, xs, s_win, 0, b_valid, lane);
        __syncwarp();                                    // staged samples consumed
        const int64_t ra = cur.row * ld, rb = ra + ld;
        const float* sa = S + cur.row * ld_s;
        PairInfo nxt{0, 0, 0};
        if (STAGE_T) {
            // the pair's S rows take the sample region's place (bulk copy; they land during the first transform) and the
            // next pair's samples are staged after the phase update instead -- they have the inverse transform's time to
            // arrive from L2 (y was written by the kernel just before).  The epilogue then reads S and tprev from shared
            // memory: no global load on the pair's critical path (ncu before: long_scoreboard 1.6 warps per issue cycle).
            if (lane == 0) {
                const uint32_t bytes = b_valid ? static_cast<uint32_t>((ld_s + kPSlot) * 4) : static_cast<uint32_t>(kPSlot * 4);
                fence_proxy_async();
                bar_expect_tx(sbar, bytes);
                bulk_g2s_hint(xs, sa, bytes, sbar, pol_keep);
            }
        } else {
            nxt = stage_next();                          // the next pair's samples have this whole pair's time to arrive
            cp_async_commit();
            const int rows = b_valid ? 2 : 1;
            warp_prefetch_l2(sa, static_cast<int>((rows - 1) * ld_s + kBins) * 4, lane);
            if (has_prev) warp_prefetch_l2(tprev + ra, static_cast<int>((rows - 1) * ld + kBins) * 8, lane);
        }
        const bool staged = STAGE_T && has_prev;
#pragma unroll 1
        for (int pass = 0; pass < 2; ++pass) {
            // ---- 1024-point forward transform: two 32-point stages around one exchange ----
#pragma unroll 1
            for (int stage = 0; stage < 2; ++stage) {
                dft32<-1>(v);
                if (stage == 0) {
                    static_for<1, 32>([&](auto k1c) {
                        constexpr int k1 = decltype(k1c)::value;
                        v[k1] = cmul(v[k1], s_tw[k1 * 32 + lane]);
                    });
                    __syncwarp();                        // pass 1: everybody has read the staged tprev rows
                    static_for<0, 32>([&](auto k1c) {
                        constexpr int k1 = decltype(k1c)::value;
                        xb[k1 * kXPitch + lane] = v[k1];
                    });
                    __syncwarp();
                    static_for<0, 32>([&](auto n2c) {
                        constexpr int n2 = decltype(n2c)::value;
                        v[n2] = xb[lane * kXPitch + n2];
                    });
                    __syncwarp();                        // tile read back
                    if (pass == 0 && staged && lane == 0) {   // pull the pair's tprev rows into the tile: they land during stage 1
                        const uint32_t bytes = b_valid ? static_cast<uint32_t>(ld * 8 + (kBins + 1) * 8) : static_cast<uint32_t>((kBins + 1) * 8);
                        fence_proxy_async();
                        bar_expect_tx(tbar, bytes);
                        bulk_g2s_hint(tile, tprev + ra, bytes, tbar, pol_stream);
                    }
                }
            }
            if (pass == 0) {
                // ---- Hermitian split, phase update; the new spectra are packed (swapped) for the second pass ----
                float2 pm[16];
                fetch_mirror(v, pm, lane);
                const float2* tsm = reinterpret_cast<const float2*>(tile);   // staged rows: a at [0, 514), b at [ld, ld + 514)
                if (staged) { bar_wait(tbar, tphase); tphase ^= 1; }
                if (STAGE_T) { bar_wait(sbar, sphase); sphase ^= 1; }
                const float* ssa = STAGE_T ? xs : sa;    // S rows: staged (row b at ld_s floats) or global
                const float* ssb = ssa + ld_s;
                float nyq_a = 0.f, nyq_b = 0.f;
                if (lane == 0) {   // bin 512 first: v[16] is overwritten below.  X[512] = 2 * Z'[512] (window carries 1/2)
                    const float2 xa = make_float2(2.f * v[16].x, 0.f), xbv = make_float2(2.f * v[16].y, 0.f);
                    const float2 z = make_float2(0.f, 0.f);
                    const float2 ta = !has_prev ? z : (staged ? tsm[512] : tprev[ra + 512]);
                    nyq_a = phase_of_rsqrt(xa, ssa[512], ta, alpha, has_prev).x;
                    st_hint(tprev + ra + 512, xa, pol_stream);
                    if (b_valid) {
                        const float2 tb = !has_prev ? z : (staged ? tsm[ld + 512] : tprev[rb + 512]);
                        nyq_b = phase_of_rsqrt(xbv, ssb[512], tb, alpha, has_prev).x;
                        st_hint(tprev + rb + 512, xbv, pol_stream);
                    }
                }
                static_for<0, 4>([&](auto gc) {
                    constexpr int g = decltype(gc)::value;
                    float2 tpa[4], tpb[4];
                    float s_a[4], s_b[4];
                    static_for<0, 4>([&](auto qc) {
                        constexpr int q = decltype(qc)::value;
                        const int k = lane + 32 * (4 * g + q);
                        s_a[q] = ssa[k];
                        s_b[q] = b_valid ? ssb[k] : 0.f;
                        if (staged) {
                            tpa[q] = tsm[k];
                            tpb[q] = b_valid ? tsm[ld + k] : make_float2(0.f, 0.f);
                        } else {
                            tpa[q] = has_prev ? tprev[ra + k] : make_float2(0.f, 0.f);
                            tpb[q] = (has_prev && b_valid) ? tprev[rb + k] : make_float2(0.f, 0.f);
                        }
                    });
                    static_for<0, 4>([&](auto qc) {
                        constexpr int q = decltype(qc)::value;
                        constexpr int k2 = 4 * g + q;
                        const int k = lane + 32 * k2;
                        float2 xa, xbv;
                        split_pair_prescaled(v[k2], pm[k2], xa, xbv);
                        float2 a = phase_of_rsqrt(xa, s_a[q], tpa[q], alpha, has_prev);
                        float2 b = make_float2(0.f, 0.f);
                        st_hint(tprev + ra + k, xa, pol_stream);
                        if (b_valid) {
                            b = phase_of_rsqrt(xbv, s_b[q], tpb[q], alpha, has_prev);
                            st_hint(tprev + rb + k, xbv, pol_stream);
                        }
                        if (k2 == 0 && lane == 0) { a.y = 0.f; b.y = 0.f; }   // irfft ignores Im(DC)
                        // V = A + iB and its mirror conj(A) + i conj(B), both with swapped components
                        v[k2] = make_float2(a.y + b.x, a.x - b.y);
                        pm[k2] = make_float2(b.x - a.y, a.x + b.y);
                    });
                });
                static_for<0, 16>([&](auto ic) {
                    constexpr int ii = decltype(ic)::value;
                    float2 r;
                    r.x = __shfl_sync(0xffffffffu, pm[15 - ii].x, pl);
                    r.y = __shfl_sync(0xffffffffu, pm[15 - ii].y, pl);
                    if (lane == 0) {
                        if constexpr (ii == 0) r = make_float2(nyq_b, nyq_a);   // irfft ignores Im(Nyquist)
                        else r = pm[16 - ii];
                    }
                    v[16 + ii] = r;
                });
                if (STAGE_T) {                           // S rows consumed: the region takes the next pair's samples
                    __syncwarp();
                    nxt = stage_next();
                    cp_async_commit();
                }
            } else {
                // ---- v = swap(ifft): frame a in .y, frame b in .x.  Hann / 1024 = s_win / 512 exactly; overlap-add of the
                // pair (frame b = frame a shifted by 8 rows of 32 samples: the same lane) ----
                static_for<0, 32>([&](auto kc) {
                    constexpr int k2 = decltype(kc)::value;
                    const float w = s_win[lane + 32 * k2] * (1.0f / 512.0f);
                    v[k2].y *= w;
                    v[k2].x = b_valid ? v[k2].x * w : 0.f;
                });
                float* seg = seg_base + 2 * ra + lane;
                static_for<0, 40>([&](auto jc) {
                    constexpr int j = decltype(jc)::value;
                    if constexpr (j < 8) st_hint(seg + 32 * j, v[j].y, pol_keep);
                    else if constexpr (j < 32) st_hint(seg + 32 * j, v[j].y + v[j - 8].x, pol_keep);
                    else { if (b_valid) st_hint(seg + 32 * j, v[j - 8].x, pol_keep); }
                });
            }
        }
        __syncwarp();
        cur = nxt;
    }
}

// ---------------------------------------------------------------------------------------
// K4: ISTFT with gather overlap-add and window-sum-square normalisation
//
// Output chunk c (samples [256c, 256c + 256) of the item) sums frames c-1 .. c+2 that exist.  An item of L = hi - lo
// samples (librosa's istft(length=L)) has ceil(L / 256) chunks: 0 .. T-2 for the default L = (T-1)*256, and beyond
// that chunk T-1 (frames T-2, T-1), chunk T (frame T-1) and later chunks with no frame, written as 0; all of these take
// the per-sample edge normalisation.  Only the item's last chunk can be partial, and only its stores are masked.
// ---------------------------------------------------------------------------------------
// BULK: a warp's two spectrum rows (8,272 B) arrive in its region by ONE bulk asynchronous copy instead of 34 scattered
// 8-byte loads per lane (ncu r01: lg_throttle 1.2 + long_scoreboard 1.7 warps per issue cycle on those loads): no LSU
// queue pressure, and all 16 warps' rows are in flight at once.
template <bool BULK>
__global__ void __launch_bounds__(kThreads, 1)
k_istft(BatchView bv, const float2* __restrict__ spec, int64_t ld, float* __restrict__ y,
        const float2* __restrict__ g_tw, const float* __restrict__ g_win) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* s_tw = reinterpret_cast<float2*>(smem_raw);
    float* s_win = reinterpret_cast<float*>(s_tw + 1024);
    spev_tile* s_ring = reinterpret_cast<spev_tile*>(s_win + 1024);
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_ring + kRing);   // one mbarrier per warp (BULK)
    int* s_tick = reinterpret_cast<int*>(s_bar + kWarps);     // [kRing] tile index held by each ring slot, -1: none
    float* s_iw = reinterpret_cast<float*>(s_tick + kRing);   // [256] 1 / sum_q w^2 for interior chunks
    float* s_x = s_iw + kHop;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    load_tables(s_tw, s_win, g_tw, g_win, 1.0f);
    if (BULK && threadIdx.x < kWarps) bar_init(s_bar + threadIdx.x, 1);
    if (BULK && threadIdx.x == 0) asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    uint64_t* tbar = s_bar + warp;
    unsigned tphase = 0;
    __syncthreads();
    for (int s = threadIdx.x; s < kHop; s += blockDim.x) {
        float wss = 0.f;   // same ascending-frame fmaf chain as the edge path below
#pragma unroll
        for (int q = 0; q < 4; ++q) { const float w = s_win[768 - 256 * q + s]; wss = fmaf(w, w, wss); }
        s_iw[s] = 1.0f / wss;
    }
    float* xw = s_x + warp * kWarpRegionWords;
    const int pl = (32 - lane) & 31;

    const int stride = gridDim.x;
    pdl_launch_dependents();
    // slot j of the ring <- the CTA's j-th tile, blockIdx.x + j * grid (thread 0 only)
    auto claim = [&](int j) {
        if (threadIdx.x != 0) return;
        int t = -1;
        const int64_t q = blockIdx.x + static_cast<int64_t>(j) * stride;
        if (q < bv.n_ctiles) t = static_cast<int>(q);
        s_tick[j & 3] = t;
        if (t >= 0) fetch_desc(s_ring + (j & 3), bv.ctiles + t);
    };
    pdl_wait();   // the spectra come from the previous kernel
    for (int j = 0; j < 3; ++j) claim(j);
    cp_async_commit();

    for (int i = 0;; ++i) {
        cp_async_wait_all();
        __syncthreads();   // previous tile's gather finished; descriptor i visible
        if (s_tick[i & 3] < 0) break;
        const spev_tile d = s_ring[i & 3];
        claim(i + 3);
        cp_async_commit();
        const int c0 = d.t0, T = d.T, nchunks = d.n;
        const int lfa = 2 * warp;
        // local frame lf <-> item frame t = c0 - 1 + lf ; needed: lf in [0, nchunks + 3)
        const int ta = c0 - 1 + lfa, tb = ta + 1;
        const bool a_valid = lfa < nchunks + 3 && ta >= 0 && ta < T;
        const bool b_valid = lfa + 1 < nchunks + 3 && tb >= 0 && tb < T;
        if (BULK && (a_valid || b_valid) && lane == 0) {      // rows a, b -> region[0 ..], region[ld ..] (float2 units)
            const uint32_t bytes = (a_valid && b_valid) ? static_cast<uint32_t>(ld * 8 + (kBins + 1) * 8)
                                                        : static_cast<uint32_t>((kBins + 1) * 8);
            const int64_t first_row = a_valid ? 0 : 1;
            fence_proxy_async();                              // the region was last read by the gather (generic proxy)
            bar_expect_tx(tbar, bytes);
            bulk_g2s(reinterpret_cast<float2*>(xw) + first_row * ld, spec + (d.row0 + lfa + first_row) * ld, bytes, tbar);
        }
        if (s_tick[(i + 1) & 3] >= 0) {   // pull the next tile's spectra of this warp into L2 during this tile's FFT
            const spev_tile& nx = s_ring[(i + 1) & 3];
            const int nta = nx.t0 - 1 + lfa;
            int r0 = lfa, r1 = lfa + 2;                       // local rows [r0, r1) to prefetch
            if (nta < 0) r0 += 1;
            if (r1 > nx.n + 3) r1 = nx.n + 3;
            if (nta + (r1 - lfa) > nx.T) r1 = lfa + (nx.T - nta);
            if (r1 > r0)
                warp_prefetch_l2(spec + (nx.row0 + r0) * ld, static_cast<int>((r1 - r0 - 1) * ld + kBins) * 8, lane);
        }

        if (a_valid || b_valid) {
            const float2* A = BULK ? reinterpret_cast<const float2*>(xw) : spec + (d.row0 + lfa) * ld;
            const float2* B = A + ld;
            if (BULK) { bar_wait(tbar, tphase); tphase ^= 1; }
            float2 v[32];
            float2 m[16];
            static_for<0, 16>([&](auto jc) {
                constexpr int j = decltype(jc)::value;
                const int k = 32 * j + lane;
                float2 a = a_valid ? A[k] : make_float2(0.f, 0.f);
                float2 b = b_valid ? B[k] : make_float2(0.f, 0.f);
                if (j == 0 && lane == 0) { a.y = 0.f; b.y = 0.f; }   // irfft ignores Im(DC)
                v[j] = make_float2(a.x - b.y, a.y + b.x);            // A + iB
                m[j] = make_float2(a.x + b.y, b.x - a.y);            // conj(A) + i conj(B)
            });
            // bins 512..1023 of the packed spectrum come from the mirror lane
            const float nyq_a = a_valid ? A[512].x : 0.f;            // irfft ignores Im(Nyquist)
            const float nyq_b = b_valid ? B[512].x : 0.f;
            static_for<0, 16>([&](auto ic) {
                constexpr int ii = decltype(ic)::value;
                float2 r;
                r.x = __shfl_sync(0xffffffffu, m[15 - ii].x, pl);
                r.y = __shfl_sync(0xffffffffu, m[15 - ii].y, pl);
                if (lane == 0) {
                    if constexpr (ii == 0) r = make_float2(nyq_a, nyq_b);
                    else r = m[16 - ii];
                }
                v[16 + ii] = r;
            });
            warp_fft1024<1>(v, reinterpret_cast<float2*>(xw), s_tw, lane);
            __syncwarp();   // transpose tile dead -> reuse for the two windowed real frames
            static_for<0, 32>([&](auto kc) {
                constexpr int k2 = decltype(kc)::value;
                const int nn = lane + 32 * k2;
                const float w = s_win[nn] * (1.0f / kNfft);
                xw[nn] = v[k2].x * w;
                xw[kNfft + nn] = v[k2].y * w;
            });
        }
        __syncthreads();
        // gather: chunk c = c0 + cl receives frames c-1, c, c+1, c+2 (ascending), local cl..cl+3.  The item's output
        // bound hi may end inside its last chunk: only that chunk stores fewer than kHop samples.
        for (int cl = warp; cl < nchunks; cl += kWarps) {
            const int c = c0 + cl;
            float* yo_c = y + d.src0 + static_cast<int64_t>(cl) * kHop;
            const int nv = static_cast<int>(min(static_cast<int64_t>(kHop), d.hi - d.src0 - static_cast<int64_t>(cl) * kHop));
            if (c >= 1 && c + 2 < T) {   // all four frames exist: table-driven normalisation
                const float* f0 = s_x + (cl >> 1) * kWarpRegionWords + (cl & 1) * kNfft + lane;
                const float* f1 = s_x + ((cl + 1) >> 1) * kWarpRegionWords + ((cl + 1) & 1) * kNfft + lane;
                const float* f2 = s_x + ((cl + 2) >> 1) * kWarpRegionWords + ((cl + 2) & 1) * kNfft + lane;
                const float* f3 = s_x + ((cl + 3) >> 1) * kWarpRegionWords + ((cl + 3) & 1) * kNfft + lane;
#pragma unroll
                for (int ii = 0; ii < kHop / 32; ++ii) {
                    const int o = 32 * ii;
                    const float sum = ((f0[768 + o] + f1[512 + o]) + f2[256 + o]) + f3[o];
                    if (lane + o < nv) yo_c[lane + o] = sum * s_iw[lane + o];
                }
                continue;
            }
#pragma unroll
            for (int ii = 0; ii < kHop / 32; ++ii) {
                const int s = lane + 32 * ii;
                float sum = 0.f, wss = 0.f;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int t = c - 1 + q;
                    if (t >= 0 && t < T) {
                        const int lf = cl + q;
                        const int nn = 768 - 256 * q + s;
                        sum += s_x[(lf >> 1) * kWarpRegionWords + (lf & 1) * kNfft + nn];
                        const float w = s_win[nn];
                        wss = fmaf(w, w, wss);
                    }
                }
                if (s < nv) yo_c[s] = wss > kTiny ? sum / wss : sum;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// K4p: overlap-add of PAIR segments (the fused Griffin-Lim iteration)
//
// k_gl_fused leaves, for every frame pair (2j, 2j+1) of an item, the 1280-sample sum of its two
// windowed inverse-transform frames at row (item row + 2j) of the `ang` workspace (float view, 2 * ld floats per row;
// a lone last frame leaves its 1024 samples).  Padded chunk q = c + 2 of output chunk c lies in the segments of pairs
// j with 0 <= q - 2j <= 4 -- two or three of them --, summed here in ascending pair order and normalised by the
// window-sum-square exactly as k_istft does (table for interior chunks, per-sample sum over the existing frames at
// the item edges).  One warp per chunk, 16-byte loads and stores, no shared-memory staging: a pure streaming kernel.
// An item longer than (T-1)*256 samples (chunk tile bound hi) also has chunk T-1 (frames T-2, T-1: pairs covering
// them are selected by the same rule, a lone last frame included) and chunk T (frame T-1 alone); later chunks meet no
// segment and are written as 0.  Only the item's last chunk can be partial; it stores sample by sample.
// ---------------------------------------------------------------------------------------
constexpr int kOlaWarps = 8;
constexpr int kOlaPerWarp = 1;                                           // chunks per warp (2 measured: no gain)
constexpr int kOlaParts = (kTileChunks + kOlaWarps * kOlaPerWarp - 1) / (kOlaWarps * kOlaPerWarp);   // CTAs per chunk tile

__global__ void __launch_bounds__(kOlaWarps * 32)
k_ola_pairs(BatchView bv, const float* __restrict__ seg, int64_t ld_f, float* __restrict__ y,
            const float* __restrict__ g_win /* [1024] Hann, then [256] 1 / sum_q w^2 (ctx table) */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float* g_iw = g_win + kNfft;
    pdl_launch_dependents();
    const int tile = blockIdx.x / kOlaParts, cl0 = ((blockIdx.x % kOlaParts) * kOlaWarps + warp) * kOlaPerWarp;
    const spev_tile* d = bv.ctiles + tile;
    const int n = __ldg(&d->n);
    if (cl0 >= n) return;
    const int t0 = __ldg(&d->t0), T = __ldg(&d->T);
    const int64_t item_row = __ldg(&d->row0) - t0 + 1;
    const int64_t src0 = __ldg(&d->src0);
    float* yo0 = y + src0;
    // the item's output bound hi ends inside this warp's chunks: kept as one predicate, the exact count is re-read from
    // the descriptor only on that path
    const bool bounded_tail = __ldg(&d->hi) - src0 - static_cast<int64_t>(cl0) * kHop < kOlaPerWarp * kHop;
    const int n_pairs = (T + 1) >> 1;
    const int s0 = 4 * lane, s1 = 128 + 4 * lane;
    pdl_wait();   // the segments come from the previous kernel
    float4 p0[kOlaPerWarp][3], p1[kOlaPerWarp][3];
#pragma unroll
    for (int e = 0; e < kOlaPerWarp; ++e) {
        const int c = t0 + cl0 + e;
        const int jlo = max(0, (c - 1) >> 1), jhi = min(n_pairs - 1, (c + 2) >> 1);
#pragma unroll
        for (int u = 0; u < 3; ++u) {
            const int j = jlo + u;
            const int off = (c + 2 - 2 * j) * kHop;
            // a lone last frame (2j + 1 == T) has no fifth chunk
            const bool ok = cl0 + e < n && j <= jhi && !(off == kNfft && 2 * j + 1 >= T);
            p0[e][u] = p1[e][u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ok) {
                const float4* src = reinterpret_cast<const float4*>(seg + (item_row + 2 * j) * ld_f + off);
                p0[e][u] = src[lane];
                p1[e][u] = src[32 + lane];
            }
        }
    }
    auto add3 = [](const float4 (&p)[3]) {
        return make_float4((p[0].x + p[1].x) + p[2].x, (p[0].y + p[1].y) + p[2].y, (p[0].z + p[1].z) + p[2].z,
                           (p[0].w + p[1].w) + p[2].w);
    };
#pragma unroll
    for (int e = 0; e < kOlaPerWarp; ++e) {
        if (cl0 + e >= n) break;
        const int c = t0 + cl0 + e;
        float4 r0 = add3(p0[e]), r1 = add3(p1[e]);
        if (c >= 1 && c + 2 < T) {
            // 1 / sum w^2 (constant table) read here, not before the wait: held across the segment loads it would take the
            // registers the masked tail stores need, and 52 instead of 48 registers cost one 256-thread CTA per SM
            const float4 w0 = __ldg(reinterpret_cast<const float4*>(g_iw + s0)), w1 = __ldg(reinterpret_cast<const float4*>(g_iw + s1));
            r0 = make_float4(r0.x * w0.x, r0.y * w0.y, r0.z * w0.z, r0.w * w0.w);
            r1 = make_float4(r1.x * w1.x, r1.y * w1.y, r1.z * w1.z, r1.w * w1.w);
        } else {
            auto norm = [&](float sum, int s) {
                float wss = 0.f;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int t = c - 1 + q;
                    if (t >= 0 && t < T) { const float w = __ldg(g_win + 768 - 256 * q + s); wss = fmaf(w, w, wss); }
                }
                return wss > kTiny ? sum / wss : sum;
            };
            r0 = make_float4(norm(r0.x, s0), norm(r0.y, s0 + 1), norm(r0.z, s0 + 2), norm(r0.w, s0 + 3));
            r1 = make_float4(norm(r1.x, s1), norm(r1.y, s1 + 1), norm(r1.z, s1 + 2), norm(r1.w, s1 + 3));
        }
        float* yo = yo0 + static_cast<int64_t>(cl0 + e) * kHop;
        if (!bounded_tail && (reinterpret_cast<uintptr_t>(yo) & 15) == 0) {   // y is read back by the next kernel: keep it in L2
            const uint64_t pol = l2_policy_evict_last();
            asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;\n" ::"l"(reinterpret_cast<float4*>(yo) + lane),
                         "f"(r0.x), "f"(r0.y), "f"(r0.z), "f"(r0.w), "l"(pol) : "memory");
            asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;\n" ::"l"(reinterpret_cast<float4*>(yo) + 32 + lane),
                         "f"(r1.x), "f"(r1.y), "f"(r1.z), "f"(r1.w), "l"(pol) : "memory");
        } else {   // unaligned, or the item's partial last chunk
            int nv = kHop;                       // samples of this chunk inside the item's output
            if (bounded_tail) {
                const spev_tile* dt = bv.ctiles + blockIdx.x / kOlaParts;
                nv = static_cast<int>(max(static_cast<int64_t>(0), min(static_cast<int64_t>(kHop),
                                                                      __ldg(&dt->hi) - __ldg(&dt->src0) - static_cast<int64_t>(cl0 + e) * kHop)));
            }
            if (s0 < nv) yo[s0] = r0.x;
            if (s0 + 1 < nv) yo[s0 + 1] = r0.y;
            if (s0 + 2 < nv) yo[s0 + 2] = r0.z;
            if (s0 + 3 < nv) yo[s0 + 3] = r0.w;
            if (s1 < nv) yo[s1] = r1.x;
            if (s1 + 1 < nv) yo[s1 + 1] = r1.y;
            if (s1 + 2 < nv) yo[s1 + 2] = r1.z;
            if (s1 + 3 < nv) yo[s1 + 3] = r1.w;
        }
    }
}

// ---------------------------------------------------------------------------------------
// Griffin-Lim initial state: ang = S * exp(i * phase)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

__global__ void k_gl_init(const float* __restrict__ S, int64_t ld_s, const float* __restrict__ phase,
                          uint64_t seed, float2* __restrict__ ang, int64_t ld, int64_t n_frames) {
    pdl_launch_dependents();
    pdl_wait();
    const int64_t total = n_frames * kBins;
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t f = i / kBins;
        const int k = static_cast<int>(i - f * kBins);
        float sn, cs;
        if (phase) {
            sincosf(phase[i], &sn, &cs);
        } else {
            const uint64_t r = splitmix64(seed ^ splitmix64(static_cast<uint64_t>(i)));
            const float u = static_cast<float>(r >> 40) * (1.0f / 16777216.0f);   // [0,1)
            sincospif(2.0f * u, &sn, &cs);
        }
        const float s = S[f * ld_s + k];
        ang[f * ld + k] = make_float2(s * cs, s * sn);
    }
}

// ---------------------------------------------------------------------------------------
// K3 (FFMA version): S = sqrt(max(pinv . mel, 0))
// ---------------------------------------------------------------------------------------
constexpr int kMagFrames = 16;
__global__ void __launch_bounds__(256)
k_mel_to_mag(BatchView bv, const float* __restrict__ mel, int layout, int is_log,
             const float* __restrict__ pinv_t /*[n_mels, 520]*/, int n_mels,
             float* __restrict__ S, int64_t ld_s) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* s_m = reinterpret_cast<float*>(smem_raw);   // [kMagFrames][n_mels]
    for (int tile = blockIdx.x; tile < bv.n_ftiles; tile += gridDim.x) {
        const spev_tile d = bv.ftiles[tile];
        const int t0 = d.t0, T = d.T, nf = d.n;
        const int64_t fo = d.row0 - t0;   // first row of the item
        for (int h0 = 0; h0 < nf; h0 += kMagFrames) {
            const int nh = min(kMagFrames, nf - h0);
            __syncthreads();
            for (int i = threadIdx.x; i < kMagFrames * n_mels; i += blockDim.x) {
                int f, m;
                if (layout == 0) { f = i / n_mels; m = i - f * n_mels; }
                else { m = i / kMagFrames; f = i - m * kMagFrames; }
                float val = 0.f;
                if (f < nh) {
                    const int t = t0 + h0 + f;
                    val = layout == 0 ? mel[(fo + t) * n_mels + m]
                                      : mel[fo * n_mels + static_cast<int64_t>(m) * T + t];
                    if (is_log) val = expf(val);
                }
                s_m[f * n_mels + m] = val;
            }
            __syncthreads();
            for (int k = threadIdx.x; k < kBins; k += blockDim.x) {
                float acc[kMagFrames];
#pragma unroll
                for (int f = 0; f < kMagFrames; ++f) acc[f] = 0.f;
                for (int m = 0; m < n_mels; ++m) {
                    const float pv = __ldg(pinv_t + m * kSpecLd + k);
#pragma unroll
                    for (int f = 0; f < kMagFrames; ++f) acc[f] = fmaf(pv, s_m[f * n_mels + m], acc[f]);
                }
#pragma unroll
                for (int f = 0; f < kMagFrames; ++f)
                    if (f < nh) S[(d.row0 + h0 + f) * ld_s + k] = sqrtf(fmaxf(acc[f], 0.f));
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// host-side launchers
// ---------------------------------------------------------------------------------------
static size_t smem_common() { return sizeof(float2) * 1024 + sizeof(float) * 1024 + sizeof(spev_tile) * kRing; }
static size_t smem_gl_fused() { return sizeof(float2) * 1024 + sizeof(float) * 1024 + sizeof(uint64_t) * 2 * kWarps + sizeof(float) * kWarps * kWsRegionWords; }
static size_t smem_ws_phase() { return sizeof(float2) * 1024 + sizeof(float) * 1024 + sizeof(uint64_t) * kWarps + sizeof(float) * kWarps * kWsRegionWords; }
static size_t smem_prog(const spev_ctx* c) { return sizeof(float4) * c->prog_groups + sizeof(int4) * kWarps * c->prog_nb; }
static size_t smem_stft(size_t prog_bytes) {
    return smem_common() + sizeof(float) * 2 * kStageSamples + sizeof(float) * kWarps * kWarpRegionWords + prog_bytes;
}
static size_t smem_istft() { return smem_common() + sizeof(uint64_t) * kWarps + sizeof(int) * kRing + sizeof(float) * kHop + sizeof(float) * kWarps * kWarpRegionWords; }

// Launch with the programmatic-stream-serialization attribute (PDL).
template <class... KArgs, class... Args>
static int launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(static_cast<unsigned>(block));
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SPEV_CUDA(cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...));
    return SPEV_OK;
}

template <class K>
static int set_smem(K kernel, size_t bytes) {
    SPEV_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(bytes)));
    return SPEV_OK;
}

static int check_batch(const spev_ctx* ctx, const spev_batch* b, bool need_ctiles) {
    SPEV_REQUIRE(ctx && b, SPEV_E_INVALID, "null ctx or batch");
    SPEV_REQUIRE(b->n_items >= 0 && b->n_frames >= 0 && b->n_ftiles >= 0 && b->n_ctiles >= 0, SPEV_E_INVALID,
                 "negative batch sizes");
    SPEV_REQUIRE(b->n_ftiles == 0 || b->ftiles, SPEV_E_INVALID, "batch.ftiles missing");
    SPEV_REQUIRE(!need_ctiles || b->n_ctiles == 0 || b->ctiles, SPEV_E_INVALID, "batch.ctiles missing");
    SPEV_REQUIRE((reinterpret_cast<uintptr_t>(b->ftiles) & 15) == 0 && (reinterpret_cast<uintptr_t>(b->ctiles) & 15) == 0,
                 SPEV_E_INVALID, "tile tables must be 16-byte aligned");
    return SPEV_OK;
}

int launch_stft_mel(spev_ctx* ctx, const spev_batch* b, const float* samples, float* out,
                    bool power_only, int log_mode, float floor_v, float lo, float hi,
                    cudaStream_t st) {
    int rc = check_batch(ctx, b, false);
    if (rc) return rc;
    if (b->n_ftiles == 0) return SPEV_OK;
    SPEV_REQUIRE(samples && out, SPEV_E_INVALID, "null samples/out");
    MelProgram mb{ctx->n_mels, ctx->prog_nb, ctx->prog_groups, ctx->d_prog_w, ctx->d_prog_h};
    const size_t smem = smem_stft(power_only ? 0 : smem_prog(ctx));
    SPEV_REQUIRE(smem <= 232448, SPEV_E_UNSUPPORTED,
                 "this mel basis (n_mels=%d: %d float4 weight groups) does not fit the fused kernel's shared memory "
                 "(%zu B > 232448); bands wider than ~128 bins (n_mels below ~24 at 22 kHz) are not supported",
                 ctx->n_mels, ctx->prog_groups, smem);
    const int grid = std::min<int64_t>(b->n_ftiles, ctx->num_sms);
    auto go = [&](auto kernel, bool mel) -> int {
        kernel<<<grid, kThreads, smem, st>>>(view_of(b), samples, out, ctx->d_tw, ctx->d_window, mb, mel ? log_mode : 0,
                                             mel ? floor_v : 0.f, mel ? lo : 0.f, mel ? hi : 0.f);
        SPEV_CUDA(cudaGetLastError());
        return SPEV_OK;
    };
    if (power_only) return go(k_stft_mel<1, 0>, false);
#define SPEV_K1_CASE(NBV) case NBV: return go(k_stft_mel<0, NBV>, true)
    switch (mb.nb) {
        SPEV_K1_CASE(1); SPEV_K1_CASE(2); SPEV_K1_CASE(3); SPEV_K1_CASE(4);
        SPEV_K1_CASE(5); SPEV_K1_CASE(6); SPEV_K1_CASE(7); SPEV_K1_CASE(8);
        default: return go(k_stft_mel<0, 0>, true);
    }
#undef SPEV_K1_CASE
}

// Grid of the persistent FFT kernels for n work tiles (also used by the Griffin-Lim driver to compute ticket bases).
int fft_grid(const spev_ctx* ctx, int64_t n_tiles) { return static_cast<int>(std::min<int64_t>(n_tiles, ctx->num_sms)); }

int launch_stft_phase(spev_ctx* ctx, const spev_batch* b, const float* y, const float* S,
                      int64_t ld_s, void* ang, void* tprev, int64_t ld, float alpha, int has_prev,
                      bool phase, cudaStream_t st, unsigned* counter, unsigned base, bool fuse) {
    int rc = check_batch(ctx, b, false);
    if (rc) return rc;
    if (b->n_ftiles == 0) return SPEV_OK;
    SPEV_REQUIRE(ang && ld >= kBins, SPEV_E_INVALID, "stft: null buffer or ld < 513");
    SPEV_REQUIRE(y || b->n_frames == b->n_items, SPEV_E_INVALID, "stft: y is null");
    if (!y) y = reinterpret_cast<const float*>(ang);   // every item has T == 1 (empty signal): never dereferenced as signal
    const int grid = fft_grid(ctx, b->n_ftiles);
    const float2* tw = ctx->d_tw;
    const float* win = ctx->d_window;
    if (!phase) {
        // plain STFT: warp-independent kernel (r01: 18.0 vs 19.9 us at cfg3, 128 vs 156 us on 120 k frames)
        return launch_pdl(k_stft_phase_w<0, false>, grid, kThreads, smem_ws_phase(), st, view_of(b), y, static_cast<const float*>(nullptr),
                          static_cast<int64_t>(0), static_cast<float2*>(ang), static_cast<float2*>(nullptr), ld, 0.f, 0, tw, win);
    }
    SPEV_REQUIRE(S && tprev && ld_s >= kBins, SPEV_E_INVALID, "phase update: null S/tprev");
    // bulk staging of the tprev rows needs 16-byte aligned rows with one readable pad column, and both rows of a pair
    // must fit the warp's transpose tile
    const bool stage_t = (reinterpret_cast<uintptr_t>(tprev) & 15) == 0 && ld % 2 == 0 && ld > kBins &&
                         static_cast<size_t>(ld) * 8 + (kBins + 1) * 8 <= sizeof(float) * kXWords;
    if (fuse) {
        // fused iteration: the new spectra are inverse-transformed in registers and leave as pair segments in `ang`
        SPEV_REQUIRE((reinterpret_cast<uintptr_t>(ang) & 15) == 0 && ld % 2 == 0 && ld * 2 >= kNfft, SPEV_E_INVALID,
                     "fused phase update: segment rows need 16-byte alignment and >= 1024 floats per row");
        // dynamic pair tickets pay once a warp has many pairs (measured: 0.72 vs 0.67 of the roofline on 138 k frames,
        // 0.635 vs 0.65 at cfg3's 2.7 pairs per warp): chosen from the batch alone, so every launch of a call agrees
        if (b->n_ftiles < 8 * grid) counter = nullptr;
        // bulk staging of the S rows: 16-byte aligned rows, both rows (+ 3 pad columns) inside the 1280-float sample region
        const bool stage_s = stage_t && (reinterpret_cast<uintptr_t>(S) & 15) == 0 && ld_s % 4 == 0 && ld_s >= kPSlot &&
                             ld_s + kPSlot <= kNfft + kHop;
        return launch_pdl(stage_s ? k_gl_fused<true> : k_gl_fused<false>, grid, kThreads, smem_gl_fused(), st, view_of(b), y, S,
                          ld_s, static_cast<float*>(ang), static_cast<float2*>(tprev), ld, alpha, has_prev, tw, win, counter, base);
    }
    return launch_pdl(stage_t ? k_stft_phase_w<1, true> : k_stft_phase_w<1, false>, grid, kThreads, smem_ws_phase(), st, view_of(b),
                      y, S, ld_s, static_cast<float2*>(ang), static_cast<float2*>(tprev), ld, alpha, has_prev, tw, win);
}

// Overlap-add of the pair segments the fused phase update left in `seg` (rows of 2 * ld floats) into y.
int launch_ola_pairs(spev_ctx* ctx, const spev_batch* b, const void* seg, int64_t ld, float* y, cudaStream_t st) {
    int rc = check_batch(ctx, b, true);
    if (rc) return rc;
    if (b->n_ctiles == 0) return SPEV_OK;
    SPEV_REQUIRE(seg && y, SPEV_E_INVALID, "ola: null buffer");
    return launch_pdl(k_ola_pairs, b->n_ctiles * kOlaParts, kOlaWarps * 32, 0, st, view_of(b), static_cast<const float*>(seg),
                      2 * ld, y, static_cast<const float*>(ctx->d_window));
}

int launch_istft(spev_ctx* ctx, const spev_batch* b, const void* spec, int64_t ld, float* y, cudaStream_t st) {
    int rc = check_batch(ctx, b, true);
    if (rc) return rc;
    if (b->n_ctiles == 0) return SPEV_OK;
    SPEV_REQUIRE(spec && y && ld >= kBins, SPEV_E_INVALID, "istft: null buffer or ld < 513");
    // bulk staging needs 16-byte aligned rows with one readable pad column, two rows per warp region
    const bool bulk = (reinterpret_cast<uintptr_t>(spec) & 15) == 0 && ld % 2 == 0 && ld > kBins &&
                      static_cast<size_t>(ld) * 8 + (kBins + 1) * 8 <= sizeof(float) * kWarpRegionWords;
    return launch_pdl(bulk ? k_istft<true> : k_istft<false>, fft_grid(ctx, b->n_ctiles), kThreads, smem_istft(), st, view_of(b),
                      static_cast<const float2*>(spec), ld, y, static_cast<const float2*>(ctx->d_tw), static_cast<const float*>(ctx->d_window));
}

// Opt every FFT kernel into the full shared-memory carve-out ONCE per ctx (per device) -- r01 re-issued
// cudaFuncSetAttribute before each of the 121 launches of a Griffin-Lim call.
int spectral_init(spev_ctx*) {
    const int kMax = 232448;
    int rc = SPEV_OK;
    auto opt = [&](auto kernel) { if (!rc) rc = set_smem(kernel, kMax); };
    opt(k_stft_mel<1, 0>); opt(k_stft_mel<0, 0>);
    opt(k_stft_mel<0, 1>); opt(k_stft_mel<0, 2>); opt(k_stft_mel<0, 3>); opt(k_stft_mel<0, 4>);
    opt(k_stft_mel<0, 5>); opt(k_stft_mel<0, 6>); opt(k_stft_mel<0, 7>); opt(k_stft_mel<0, 8>);
    opt(k_stft_phase_w<0, false>); opt(k_stft_phase_w<1, false>); opt(k_stft_phase_w<1, true>);
    opt(k_gl_fused<true>); opt(k_gl_fused<false>);
    opt(k_istft<true>); opt(k_istft<false>);
    return rc;
}

int launch_gl_init(spev_ctx* ctx, const float* S, int64_t ld_s, const float* phase, uint64_t seed,
                   void* ang, int64_t ld, int64_t n_frames, cudaStream_t st) {
    if (n_frames == 0) return SPEV_OK;
    const int64_t total = n_frames * kBins;
    const int grid = static_cast<int>(std::min<int64_t>((total + 255) / 256, ctx->num_sms * 16));
    int rc = launch_pdl(k_gl_init, grid, 256, 0, st, S, ld_s, phase, seed, static_cast<float2*>(ang), ld, n_frames);
    if (rc) return rc;
    return SPEV_OK;
}

int launch_mel_to_mag(spev_ctx* ctx, const spev_batch* b, const float* mel, int layout, int is_log,
                      float* S, int64_t ld_s, cudaStream_t st) {
    int rc = check_batch(ctx, b, false);
    if (rc) return rc;
    if (b->n_ftiles == 0) return SPEV_OK;
    SPEV_REQUIRE(mel && S && ld_s >= kBins, SPEV_E_INVALID, "mel_to_mag: null buffer or ld < 513");
    SPEV_REQUIRE(layout == 0 || layout == 1, SPEV_E_INVALID, "mel_to_mag: layout must be 0 or 1");
    const size_t smem = sizeof(float) * kMagFrames * ctx->n_mels;
    const int grid = std::min<int64_t>(b->n_ftiles, ctx->num_sms * 4);
    k_mel_to_mag<<<grid, 256, smem, st>>>(view_of(b), mel, layout, is_log, ctx->d_pinv_t,
                                          ctx->n_mels, S, ld_s);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

}  // namespace spev
