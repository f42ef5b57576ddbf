// lr.cu -- LengthRegulator (duration sanitise + warp-scan cumsum + gather-expand), duration
// rule and bucketize+embedding kernels for sm_100a.  All index arithmetic is integer and
// bit-exact against the reference; payload rows are copied verbatim.
//
// K6 k_lr_plan     replaces the validation loop of LengthRegulator.forward
//                  (/root/reference/spev_real_metrics.py:126-142) -- which performs one
//                  .item() device sync per (b,t) -- with one warp-scan per row.
// K7 k_lr_expand   replaces repeat/cat/pad/stack (:135-146) and the five expand_feat calls
//                  (:228-236) + post-clamps (:239-243) in the fused variant.
// K8 k_bucketize   torch.bucketize + F.embedding (SURVEY a-13; no in-tree reference site).
#include <algorithm>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "spev_internal.cuh"

namespace spev {

// ---- duration sanitisation: "if not np.isfinite(d) or d < 0 or d > 1000: d = 0; n = int(d)" ----
__device__ __forceinline__ int sanitize(long long d) { return (d < 0 || d > 1000) ? 0 : static_cast<int>(d); }
__device__ __forceinline__ int sanitize(int d) { return (d < 0 || d > 1000) ? 0 : d; }
__device__ __forceinline__ int sanitize(double d) {
    return (!isfinite(d) || d < 0.0 || d > 1000.0) ? 0 : static_cast<int>(d);   // cast truncates
}
__device__ __forceinline__ int sanitize(float d) { return sanitize(static_cast<double>(d)); }
__device__ __forceinline__ int sanitize(__half d) { return sanitize(static_cast<double>(__half2float(d))); }
__device__ __forceinline__ int sanitize(__nv_bfloat16 d) { return sanitize(static_cast<double>(__bfloat162float(d))); }

template <class Tdur>
__global__ void k_lr_plan(const Tdur* __restrict__ dur, int B, int T, int32_t* __restrict__ cumsum,
                          long long* __restrict__ mel_lens, long long* __restrict__ max_len) {
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    for (int b = blockIdx.x * warps_per_block + (threadIdx.x >> 5); b < B; b += gridDim.x * warps_per_block) {
        const Tdur* row = dur + static_cast<int64_t>(b) * T;
        int32_t* crow = cumsum + static_cast<int64_t>(b) * T;
        int carry = 0;
        for (int t0 = 0; t0 < T; t0 += 32) {
            const int t = t0 + lane;
            int v = t < T ? sanitize(row[t]) : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, v, o);
                if (lane >= o) v += u;
            }
            v += carry;
            if (t < T) crow[t] = v;
            carry = __shfl_sync(0xffffffffu, v, 31);
        }
        if (lane == 0) {
            const long long len = carry > 0 ? carry : 1;   // empty row -> one zero frame
            mel_lens[b] = len;
            atomicMax(max_len, len);
        }
    }
}

// first i in [0,T) with cs[i] > f   (np.searchsorted(cs, f, side='right')); caller guarantees
// f < cs[T-1]
__device__ __forceinline__ int upper_bound_i32(const int32_t* cs, int T, int f) {
    int lo = 0, hi = T;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (cs[mid] > f) hi = mid; else lo = mid + 1;
    }
    return lo;
}

// torch.clamp propagates NaN (the reference then reports it through its "NaN detected" guards, :255-257);
// fminf/fmaxf alone would turn a NaN into the lower bound.
__device__ __forceinline__ float clamp_nan(float v, float lo, float hi) { return v != v ? v : fminf(fmaxf(v, lo), hi); }

constexpr int kLrFrames = 64;     // output frames per CTA
constexpr int kLrThreads = 256;
constexpr int kMaxFeat = 16;
struct ClampParams { int enabled; float lo[kMaxFeat]; float hi[kMaxFeat]; };   // by-value kernel arg

// out[b, f, :] = x[b, idx, :] (row_bytes bytes) or 0; optional n_feat scalar curves.
__global__ void __launch_bounds__(kLrThreads)
k_lr_expand(const unsigned char* __restrict__ x, int64_t row_bytes, const float* __restrict__ feats,
            int n_feat, ClampParams clamp,
            const int32_t* __restrict__ cumsum, int B, int T, unsigned char* __restrict__ out,
            float* __restrict__ feats_out, int64_t max_len) {
    __shared__ int s_idx[kLrFrames];
    const int b = blockIdx.y;
    const int64_t f0 = static_cast<int64_t>(blockIdx.x) * kLrFrames;
    const int32_t* cs = cumsum + static_cast<int64_t>(b) * T;
    const int total = T > 0 ? cs[T - 1] : 0;
    if (threadIdx.x < kLrFrames) {
        const int64_t f = f0 + threadIdx.x;
        s_idx[threadIdx.x] = (f < total) ? upper_bound_i32(cs, T, static_cast<int>(f)) : -1;
    }
    __syncthreads();
    const int nfr = static_cast<int>(min(static_cast<int64_t>(kLrFrames), max_len - f0));
    const unsigned char* xb = x + static_cast<int64_t>(b) * T * row_bytes;
    unsigned char* ob = out + (static_cast<int64_t>(b) * max_len + f0) * row_bytes;

    if (x != nullptr) {
        const bool vec16 = (row_bytes % 16 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) &&
                           ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
        const bool vec4 = (row_bytes % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 3) == 0) &&
                          ((reinterpret_cast<uintptr_t>(out) & 3) == 0);
        if (vec16) {
            const int per_row = static_cast<int>(row_bytes / 16);
            const int64_t n = static_cast<int64_t>(nfr) * per_row;
            for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
                const int fl = static_cast<int>(i / per_row);
                const int c = static_cast<int>(i - static_cast<int64_t>(fl) * per_row);
                const int idx = s_idx[fl];
                uint4 v = make_uint4(0, 0, 0, 0);
                if (idx >= 0) v = __ldg(reinterpret_cast<const uint4*>(xb + idx * row_bytes) + c);
                reinterpret_cast<uint4*>(ob + fl * row_bytes)[c] = v;
            }
        } else if (vec4) {
            const int per_row = static_cast<int>(row_bytes / 4);
            const int64_t n = static_cast<int64_t>(nfr) * per_row;
            for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
                const int fl = static_cast<int>(i / per_row);
                const int c = static_cast<int>(i - static_cast<int64_t>(fl) * per_row);
                const int idx = s_idx[fl];
                uint32_t v = 0;
                if (idx >= 0) v = __ldg(reinterpret_cast<const uint32_t*>(xb + idx * row_bytes) + c);
                reinterpret_cast<uint32_t*>(ob + fl * row_bytes)[c] = v;
            }
        } else {
            const int64_t n = static_cast<int64_t>(nfr) * row_bytes;
            for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
                const int fl = static_cast<int>(i / row_bytes);
                const int64_t c = i - fl * row_bytes;
                const int idx = s_idx[fl];
                ob[i] = idx >= 0 ? xb[idx * row_bytes + c] : 0;
            }
        }
    }
    // scalar curves: thread <-> (feature j, local frame) -> coalesced in f
    for (int i = threadIdx.x; i < n_feat * nfr; i += blockDim.x) {
        const int j = i / nfr, fl = i - j * nfr;
        const int idx = s_idx[fl];
        float v = 0.f;
        if (idx >= 0) v = __ldg(feats + (static_cast<int64_t>(j) * B + b) * T + idx);
        if (clamp.enabled) v = clamp_nan(v, clamp.lo[j], clamp.hi[j]);
        feats_out[(static_cast<int64_t>(j) * B + b) * max_len + f0 + fl] = v;
    }
}

// ---- fused variance adaptor: expand + n_feat Conv1d(1->H, k=3, pad=1) embeddings + sum -----------------
// out[b,f,c] = x[b,idx(b,f),c] (0 past the row's length)
//            + sum_j ( bias_j[c] + w_j[c,0]*cv_j[b,f-1] + w_j[c,1]*cv_j[b,f] + w_j[c,2]*cv_j[b,f+1] )
// with cv_j[b,f] = clamp(curve_j[b,idx(b,f)], lo_j, hi_j) inside the row, 0 outside [0, max_len) and past
// the row's length -- i.e. spev_real_metrics.py:226-252 (six LengthRegulator calls, five clamps, five
// Conv1d embeddings, their sum) in one launch; x_expanded and the expanded curves never reach HBM.
// Thread <-> channel (weights of the thread's channel live in registers), CTA <-> 64 frames of one row.
constexpr int kVaFrames = 64;
constexpr int kVaMaxFeat = 8;
__global__ void __launch_bounds__(256)
k_variance_fuse(const float* __restrict__ x, const float* __restrict__ feats, int n_feat, ClampParams clamp,
                const float* __restrict__ conv_w /*[n_feat,H,3]*/, const float* __restrict__ conv_b /*[n_feat,H]*/,
                const int32_t* __restrict__ cumsum, int B, int T, int H, float* __restrict__ out,
                float* __restrict__ feats_out /*nullable [n_feat,B,max_len]*/, int64_t max_len) {
    __shared__ int s_idx[kVaFrames + 2];
    __shared__ float s_cv[kVaMaxFeat][kVaFrames + 2];
    const int b = blockIdx.y;
    const int64_t f0 = static_cast<int64_t>(blockIdx.x) * kVaFrames;
    const int32_t* cs = cumsum + static_cast<int64_t>(b) * T;
    const int total = T > 0 ? cs[T - 1] : 0;
    for (int i = threadIdx.x; i < kVaFrames + 2; i += blockDim.x) {
        const int64_t f = f0 - 1 + i;                         // halo of one frame on each side
        s_idx[i] = (f >= 0 && f < total) ? upper_bound_i32(cs, T, static_cast<int>(f)) : -1;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_feat * (kVaFrames + 2); i += blockDim.x) {
        const int j = i / (kVaFrames + 2), fl = i - j * (kVaFrames + 2);
        const int idx = s_idx[fl];
        const int64_t f = f0 - 1 + fl;
        float v = 0.f;
        if (idx >= 0) v = __ldg(feats + (static_cast<int64_t>(j) * B + b) * T + idx);
        // the reference clamps the zero-padded tensor: positions past the row's length hold clamp(0),
        // positions outside [0, max_len) are the convolution's zero padding
        if (clamp.enabled) v = clamp_nan(v, clamp.lo[j], clamp.hi[j]);
        if (f < 0 || f >= max_len) v = 0.f;
        s_cv[j][fl] = v;
        if (feats_out && fl >= 1 && fl <= kVaFrames && f < max_len)
            feats_out[(static_cast<int64_t>(j) * B + b) * max_len + f] = v;
    }
    __syncthreads();
    const int nfr = static_cast<int>(min(static_cast<int64_t>(kVaFrames), max_len - f0));
    const float* xb = x + static_cast<int64_t>(b) * T * H;
    float* ob = out + (static_cast<int64_t>(b) * max_len + f0) * H;
    for (int c = threadIdx.x; c < H; c += blockDim.x) {
        float w0[kVaMaxFeat], w1[kVaMaxFeat], w2[kVaMaxFeat], bs[kVaMaxFeat];
#pragma unroll
        for (int j = 0; j < kVaMaxFeat; ++j) {
            if (j < n_feat) {
                const float* w = conv_w + (static_cast<int64_t>(j) * H + c) * 3;
                w0[j] = __ldg(w); w1[j] = __ldg(w + 1); w2[j] = __ldg(w + 2);
                bs[j] = __ldg(conv_b + static_cast<int64_t>(j) * H + c);
            }
        }
        for (int fl = 0; fl < nfr; ++fl) {
            const int idx = s_idx[fl + 1];
            float acc = idx >= 0 ? __ldg(xb + static_cast<int64_t>(idx) * H + c) : 0.f;
#pragma unroll
            for (int j = 0; j < kVaMaxFeat; ++j) {
                if (j < n_feat) {
                    // one embedding: bias + 3-tap correlation, then added to the running sum in the
                    // reference's left-to-right order (dec_input + pitch + energy + breath + rough + bright)
                    float e = fmaf(w0[j], s_cv[j][fl], bs[j]);
                    e = fmaf(w1[j], s_cv[j][fl + 1], e);
                    e = fmaf(w2[j], s_cv[j][fl + 2], e);
                    acc += e;
                }
            }
            ob[static_cast<int64_t>(fl) * H + c] = acc;
        }
    }
}

// ---- backward of the expand (autograd of repeat/cat/pad/stack, spev_real_metrics.py:135-146) ----------
// grad_x[b,t,:] = sum over the frames f of segment t (cumsum[t-1] <= f < cumsum[t], f < max_len) of
// grad_out[b,f,:].  One owner thread per (b, t, VEC channels) sums its frame range in ascending order:
// no atomics, deterministic.  Padding frames (f >= total_b) belong to no segment and contribute nothing,
// like the zero rows F.pad appends in the reference.
template <class T> struct AccOf { using type = float; };
template <> struct AccOf<double> { using type = double; };
__device__ __forceinline__ float to_acc(float v) { return v; }
__device__ __forceinline__ double to_acc(double v) { return v; }
__device__ __forceinline__ float to_acc(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_acc(__nv_bfloat16 v) { return __bfloat162float(v); }
template <class T> __device__ __forceinline__ T from_acc(typename AccOf<T>::type v);
template <> __device__ __forceinline__ float from_acc<float>(float v) { return v; }
template <> __device__ __forceinline__ double from_acc<double>(double v) { return v; }
template <> __device__ __forceinline__ __half from_acc<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_acc<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

template <class T>
__global__ void __launch_bounds__(256)
k_lr_expand_bwd(const T* __restrict__ grad_out, int H, const int32_t* __restrict__ cumsum, int B, int Tn,
                int64_t max_len, T* __restrict__ grad_x) {
    using Acc = typename AccOf<T>::type;
    const int64_t n = static_cast<int64_t>(B) * Tn * H;
    for (int64_t e = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; e < n;
         e += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t bt = e / H;
        const int c = static_cast<int>(e - bt * H);
        const int b = static_cast<int>(bt / Tn), t = static_cast<int>(bt - static_cast<int64_t>(b) * Tn);
        const int32_t* cs = cumsum + static_cast<int64_t>(b) * Tn;
        const int64_t lo = t > 0 ? cs[t - 1] : 0;
        const int64_t hi = min(static_cast<int64_t>(cs[t]), max_len);
        const T* g = grad_out + (static_cast<int64_t>(b) * max_len) * H + c;
        Acc acc = 0;
        for (int64_t f = lo; f < hi; ++f) acc += to_acc(g[f * H]);
        grad_x[e] = from_acc<T>(acc);
    }
}

// float32 rows whose length is a multiple of 4: one owner thread per (b, t, float4)
__global__ void __launch_bounds__(256)
k_lr_expand_bwd_f4(const float4* __restrict__ grad_out, int H4, const int32_t* __restrict__ cumsum, int B, int Tn,
                   int64_t max_len, float4* __restrict__ grad_x) {
    const int64_t n = static_cast<int64_t>(B) * Tn * H4;
    for (int64_t e = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; e < n;
         e += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t bt = e / H4;
        const int c = static_cast<int>(e - bt * H4);
        const int b = static_cast<int>(bt / Tn), t = static_cast<int>(bt - static_cast<int64_t>(b) * Tn);
        const int32_t* cs = cumsum + static_cast<int64_t>(b) * Tn;
        const int64_t lo = t > 0 ? cs[t - 1] : 0;
        const int64_t hi = min(static_cast<int64_t>(cs[t]), max_len);
        const float4* g = grad_out + (static_cast<int64_t>(b) * max_len) * H4 + c;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int64_t f = lo; f < hi; ++f) {
            const float4 v = __ldg(g + f * H4);
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        grad_x[e] = acc;
    }
}

// scalar curves: grad_feats[j,b,t] = pass(feats[j,b,t]) * sum over segment t of grad_feats_out[j,b,f];
// pass = lo <= v <= hi (torch.clamp's backward mask; NaN does not pass), 1 when no clamp was applied.
__global__ void __launch_bounds__(256)
k_lr_curves_bwd(const float* __restrict__ grad_fo, const float* __restrict__ feats, int n_feat, ClampParams clamp,
                const int32_t* __restrict__ cumsum, int B, int Tn, int64_t max_len, float* __restrict__ grad_feats) {
    const int64_t n = static_cast<int64_t>(n_feat) * B * Tn;
    for (int64_t e = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; e < n;
         e += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t jb = e / Tn;
        const int t = static_cast<int>(e - jb * Tn);
        const int j = static_cast<int>(jb / B), b = static_cast<int>(jb - static_cast<int64_t>(j) * B);
        const int32_t* cs = cumsum + static_cast<int64_t>(b) * Tn;
        const int64_t lo = t > 0 ? cs[t - 1] : 0;
        const int64_t hi = min(static_cast<int64_t>(cs[t]), max_len);
        bool pass = true;
        if (clamp.enabled) {
            const float v = feats[e];
            pass = v >= clamp.lo[j] && v <= clamp.hi[j];
        }
        float acc = 0.f;
        if (pass) {
            const float* g = grad_fo + jb * max_len;
            for (int64_t f = lo; f < hi; ++f) acc += g[f];
        }
        grad_feats[e] = acc;
    }
}

// ---- backward of the fused variance adaptor (k_variance_fuse) ------------------------------------------
// With g = grad_out [B,maxF,H], cv_j the expanded + clamped curves (recomputed, never stored):
//   grad_b[j][c]    = sum_{b,f} g[b,f,c]                                  (same for every j)
//   grad_w[j][c][k] = sum_{b,f} g[b,f,c] * cv_j[b,f+k-1]
//   grad_cv_j[b,f]  = t_j0[b,f+1] + t_j1[b,f] + t_j2[b,f-1],   t_jk[b,f] = sum_c g[b,f,c] * w_j[c,k]
//   grad_feats[j,b,t] = sum over segment t of grad_cv_j[b,f] where the clamp passed   (k_lr_curves_bwd)
//   grad_x = segment sum of g                                                        (k_lr_expand_bwd)
// Thread <-> channel, CTA <-> a static list of 64-frame tiles (tile = blockIdx.x + i*gridDim.x): the 16 weight /
// bias partial sums stay in registers across the CTA's tiles and are written once per CTA; a second kernel adds
// the per-CTA partials in CTA order.  The per-frame sums over channels use a 16-value warp transpose-reduce
// (16 shuffles per frame instead of 75) and a fixed-order sum over the warps.  No atomics: deterministic.

// Sum 16 per-lane values over the 32 lanes of a warp; on return lane l holds (in v[0]) the warp total of value
// index slot_of(l & 15).  Fixed butterfly: the result does not depend on anything but the inputs.
__device__ __forceinline__ int reduce16_slot(int lane) {
    return ((lane & 1) << 3) | ((lane & 2) << 1) | ((lane & 4) >> 1) | ((lane & 8) >> 3);
}
__device__ __forceinline__ float warp_reduce16(float (&v)[16], int lane) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const bool up = lane & 1;
        const float send = up ? v[i] : v[i + 8], keep = up ? v[i + 8] : v[i];
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const bool up = lane & 2;
        const float send = up ? v[i] : v[i + 4], keep = up ? v[i + 4] : v[i];
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const bool up = lane & 4;
        const float send = up ? v[i] : v[i + 2], keep = up ? v[i + 2] : v[i];
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
    {
        const bool up = lane & 8;
        const float send = up ? v[0] : v[1], keep = up ? v[1] : v[0];
        v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    v[0] += __shfl_xor_sync(0xffffffffu, v[0], 16);
    return v[0];
}

template <int NF>   // number of curves (compile time: the accumulators must live in registers)
__global__ void __launch_bounds__(1024)
k_variance_fuse_bwd(const float* __restrict__ grad_out, const float* __restrict__ feats, ClampParams clamp,
                    const float* __restrict__ conv_w /*[NF,H,3]*/, const int32_t* __restrict__ cumsum, int B, int Tn,
                    int H, int64_t max_len, int tiles_per_row, float* __restrict__ grad_cv /*[NF,B,max_len]*/,
                    float* __restrict__ partials /*[gridDim.x][H][3*NF+1]*/) {
    constexpr int kF = kVaFrames + 2;              // frames f0-1 .. f0+64
    constexpr int kJK = 3 * NF;
    static_assert(kJK <= 16, "at most 5 curves per pass");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int* s_idx = reinterpret_cast<int*>(smem_raw);                 // [kF]
    float* s_cv = reinterpret_cast<float*>(s_idx + kF + 2);         // [NF][kF]
    unsigned char* s_pass = reinterpret_cast<unsigned char*>(s_cv + NF * kF);   // [NF][kF]
    float* s_t = reinterpret_cast<float*>(s_pass + ((NF * kF + 15) & ~15));     // [16][kF]
    float* s_part = s_t + 16 * kF;                                  // [kF][nwarps][16]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int c = threadIdx.x;
    const bool c_ok = c < H;
    float w[kJK];
#pragma unroll
    for (int q = 0; q < kJK; ++q) w[q] = c_ok ? __ldg(conv_w + (static_cast<int64_t>(q / 3) * H + c) * 3 + q % 3) : 0.f;
    float acc_w[kJK], acc_b = 0.f;
#pragma unroll
    for (int q = 0; q < kJK; ++q) acc_w[q] = 0.f;
    const int slot = reduce16_slot(lane);
    const int64_t n_tiles = static_cast<int64_t>(B) * tiles_per_row;

    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int b = static_cast<int>(tile / tiles_per_row);
        const int64_t f0 = (tile - static_cast<int64_t>(b) * tiles_per_row) * kVaFrames;
        const int32_t* cs = cumsum + static_cast<int64_t>(b) * Tn;
        const int total = Tn > 0 ? cs[Tn - 1] : 0;
        __syncthreads();                                   // previous tile's shared data fully consumed
        for (int i = threadIdx.x; i < kF; i += blockDim.x) {
            const int64_t f = f0 - 1 + i;
            s_idx[i] = (f >= 0 && f < total) ? upper_bound_i32(cs, Tn, static_cast<int>(f)) : -1;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < NF * kF; i += blockDim.x) {
            const int j = i / kF, fl = i - j * kF;
            const int idx = s_idx[fl];
            const int64_t f = f0 - 1 + fl;
            float v = 0.f;
            bool pass = idx >= 0;
            if (idx >= 0) v = __ldg(feats + (static_cast<int64_t>(j) * B + b) * Tn + idx);
            if (clamp.enabled) {
                pass = pass && v >= clamp.lo[j] && v <= clamp.hi[j];
                v = clamp_nan(v, clamp.lo[j], clamp.hi[j]);
            }
            if (f < 0 || f >= max_len) v = 0.f;
            s_cv[i] = v;
            s_pass[i] = pass ? 1 : 0;
        }
        __syncthreads();
        const float* gb = grad_out + (static_cast<int64_t>(b) * max_len) * H + c;
        for (int fl = 0; fl < kF; ++fl) {
            const int64_t f = f0 - 1 + fl;
            const float g = (c_ok && f >= 0 && f < max_len) ? __ldg(gb + f * H) : 0.f;
            if (fl >= 1 && fl <= kVaFrames) {              // interior frame: weight / bias partial sums
                acc_b += g;
#pragma unroll
                for (int q = 0; q < kJK; ++q) acc_w[q] = fmaf(g, s_cv[(q / 3) * kF + fl - 1 + q % 3], acc_w[q]);
            }
            float p[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) p[q] = q < kJK ? g * w[q] : 0.f;
            const float tot = warp_reduce16(p, lane);
            if (lane < 16) s_part[(fl * nwarps + warp) * 16 + slot] = tot;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < kF * 16; i += blockDim.x) {
            const int fl = i >> 4, q = i & 15;
            float s = 0.f;
            for (int wq = 0; wq < nwarps; ++wq) s += s_part[(fl * nwarps + wq) * 16 + q];
            s_t[q * kF + fl] = s;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < NF * kVaFrames; i += blockDim.x) {
            const int j = i / kVaFrames, fl = 1 + (i - j * kVaFrames);
            const int64_t f = f0 - 1 + fl;
            if (f < max_len) {
                float gcv = 0.f;
                if (s_pass[j * kF + fl])
                    gcv = (s_t[(3 * j) * kF + fl + 1] + s_t[(3 * j + 1) * kF + fl]) + s_t[(3 * j + 2) * kF + fl - 1];
                grad_cv[(static_cast<int64_t>(j) * B + b) * max_len + f] = gcv;
            }
        }
    }
    if (c_ok) {
        float* pp = partials + (static_cast<int64_t>(blockIdx.x) * H + c) * (kJK + 1);
#pragma unroll
        for (int q = 0; q < kJK; ++q) pp[q] = acc_w[q];
        pp[kJK] = acc_b;
    }
}

// grad_w[j][c][k] / grad_b[j][c] = sum of the per-CTA partials in CTA order
__global__ void k_variance_bwd_reduce(const float* __restrict__ partials, int n_part, int H, int n_feat,
                                      float* __restrict__ grad_w, float* __restrict__ grad_b) {
    const int stride = 3 * n_feat + 1;
    const int n = H * stride;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int c = i / stride, q = i - c * stride;
        float s = 0.f;
        for (int p = 0; p < n_part; ++p) s += partials[(static_cast<int64_t>(p) * H + c) * stride + q];
        if (q < 3 * n_feat) {
            if (grad_w) grad_w[(static_cast<int64_t>(q / 3) * H + c) * 3 + q % 3] = s;
        } else if (grad_b) {
            for (int j = 0; j < n_feat; ++j) grad_b[static_cast<int64_t>(j) * H + c] = s;
        }
    }
}

// ---- duration rule: clamp((exp(ld)-1)*d_control, 0, 500).round().long(), spev_real_metrics.py:215 ----
__global__ void k_duration_rule(const float* __restrict__ ld, int64_t n, float d_control,
                                long long* __restrict__ dur) {
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        // float32 exp evaluated through float64 so that the result is the correctly rounded
        // float32 value (torch CPU: SLEEF <= 1 ulp); the remaining ops are exact float32.
        const float e = static_cast<float>(exp(static_cast<double>(ld[i])));
        float v = (e - 1.0f) * d_control;
        v = fminf(fmaxf(v, 0.0f), 500.0f);
        dur[i] = static_cast<long long>(rintf(v));   // round half to even
    }
}

// ---- bucketize (+ embedding) ----
__device__ __forceinline__ int bucket_of(float v, const float* __restrict__ bnd, int nb, int right) {
    int lo = 0, hi = nb;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const float m = bnd[mid];
        // same predicates as ATen's lower/upper bound: NaN falls through to nb
        const bool go_right = right ? !(m > v) : !(m >= v);
        if (go_right) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(256)
k_bucketize_embed(const float* __restrict__ v, int64_t n, const float* __restrict__ bnd, int nb,
                  int right, const float* __restrict__ table, int H, long long* __restrict__ idx_out,
                  float* __restrict__ out, int accumulate) {
    extern __shared__ float s_bnd[];
    for (int i = threadIdx.x; i < nb; i += blockDim.x) s_bnd[i] = bnd[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    const bool vec = (H % 4 == 0) && ((reinterpret_cast<uintptr_t>(table) & 15) == 0) &&
                     ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    for (int64_t e0 = (static_cast<int64_t>(blockIdx.x) * wpb + (threadIdx.x >> 5)) * 32; e0 < n;
         e0 += static_cast<int64_t>(gridDim.x) * wpb * 32) {
        // each lane classifies one element, then the warp copies the 32 rows cooperatively
        const int64_t e = e0 + lane;
        int my = 0;
        if (e < n) {
            my = bucket_of(v[e], s_bnd, nb, right);
            if (idx_out) idx_out[e] = my;
        }
        if (out == nullptr) continue;
        const int cnt = static_cast<int>(min(static_cast<int64_t>(32), n - e0));
        for (int r = 0; r < cnt; ++r) {
            const int idx = __shfl_sync(0xffffffffu, my, r);
            const float* src = table + static_cast<int64_t>(idx) * H;
            float* dst = out + (e0 + r) * H;
            if (vec) {
                for (int c = lane; c < H / 4; c += 32) {
                    float4 t = __ldg(reinterpret_cast<const float4*>(src) + c);
                    if (accumulate) {
                        const float4 o = reinterpret_cast<float4*>(dst)[c];
                        t.x += o.x; t.y += o.y; t.z += o.z; t.w += o.w;
                    }
                    reinterpret_cast<float4*>(dst)[c] = t;
                }
            } else {
                for (int c = lane; c < H; c += 32) {
                    float t = __ldg(src + c);
                    if (accumulate) t += dst[c];
                    dst[c] = t;
                }
            }
        }
    }
}

// ---- 16-bit PCM -> float32 (x / 32768): what soundfile/librosa.load produce from a 16-bit wav ----
__global__ void k_pcm16_to_f32(const short* __restrict__ in, int64_t n, float* __restrict__ out) {
    const int64_t n8 = n >> 3;
    const bool vec = ((reinterpret_cast<uintptr_t>(in) & 15) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    const int64_t tid = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    const int64_t nthr = static_cast<int64_t>(gridDim.x) * blockDim.x;
    int64_t done = 0;
    if (vec) {
        for (int64_t i = tid; i < n8; i += nthr) {
            const int4 v = __ldg(reinterpret_cast<const int4*>(in) + i);   // 8 samples
            const int w[4] = {v.x, v.y, v.z, v.w};
            float f[8];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                f[2 * j] = static_cast<float>(static_cast<short>(w[j] & 0xffff)) * (1.0f / 32768.0f);
                f[2 * j + 1] = static_cast<float>(static_cast<short>(w[j] >> 16)) * (1.0f / 32768.0f);
            }
            float4* o = reinterpret_cast<float4*>(out) + 2 * i;
            o[0] = make_float4(f[0], f[1], f[2], f[3]);
            o[1] = make_float4(f[4], f[5], f[6], f[7]);
        }
        done = n8 << 3;
    }
    for (int64_t i = done + tid; i < n; i += nthr) out[i] = static_cast<float>(in[i]) * (1.0f / 32768.0f);
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
static void fill_clamp(ClampParams& cp, int n_feat, const float* clamp_lo, const float* clamp_hi) {
    cp.enabled = (n_feat > 0 && clamp_lo && clamp_hi) ? 1 : 0;
    for (int j = 0; j < kMaxFeat; ++j) {
        cp.lo[j] = (cp.enabled && j < n_feat) ? clamp_lo[j] : 0.f;
        cp.hi[j] = (cp.enabled && j < n_feat) ? clamp_hi[j] : 0.f;
    }
}

static int grid_for(int64_t n, int block) {
    return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((n + block - 1) / block, 148 * 16)));
}

static int va_bwd_grid(int B, int64_t max_len) {
    const int64_t tiles = static_cast<int64_t>(B) * ((max_len + kVaFrames - 1) / kVaFrames);
    return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(tiles, 148 * 2)));
}

template <int NF>
static int launch_va_bwd(const float* grad_out, const float* feats, const ClampParams& cp, const float* conv_w,
                         const int32_t* cumsum, int B, int T, int H, int64_t max_len, float* grad_cv, float* partials,
                         int grid, cudaStream_t st) {
    const int threads = (H + 31) & ~31;
    const int kF = kVaFrames + 2;
    const size_t smem = sizeof(int) * (kF + 2) + sizeof(float) * NF * kF + ((NF * kF + 15) & ~15) +
                        sizeof(float) * 16 * kF + sizeof(float) * kF * (threads / 32) * 16;
    SPEV_CUDA(cudaFuncSetAttribute(k_variance_fuse_bwd<NF>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    const int tiles_per_row = static_cast<int>((max_len + kVaFrames - 1) / kVaFrames);
    k_variance_fuse_bwd<NF><<<grid, threads, smem, st>>>(grad_out, feats, cp, conv_w, cumsum, B, T, H, max_len, tiles_per_row,
                                                         grad_cv, partials);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

}  // namespace spev

using namespace spev;

extern "C" {

int spev_pcm16_to_f32(const int16_t* pcm, int64_t n, float* out, void* stream) {
    SPEV_REQUIRE(n >= 0, SPEV_E_INVALID, "pcm16_to_f32: n < 0");
    if (n == 0) return SPEV_OK;
    SPEV_REQUIRE(pcm && out, SPEV_E_INVALID, "pcm16_to_f32: null buffer");
    const int grid = static_cast<int>(std::min<int64_t>((n / 8 + 255) / 256 + 1, 148 * 16));
    k_pcm16_to_f32<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const short*>(pcm), n, out);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

int spev_lr_plan(const void* dur, int dur_dtype, int B, int T, int32_t* cumsum, int64_t* mel_lens,
                 int64_t* max_len_dev, int64_t* max_len_host, void* stream) {
    SPEV_REQUIRE(B >= 0 && T >= 0, SPEV_E_INVALID, "lr_plan: negative shape");
    SPEV_REQUIRE(max_len_dev, SPEV_E_INVALID, "lr_plan: max_len_dev is null");
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    SPEV_CUDA(cudaMemsetAsync(max_len_dev, 0, sizeof(int64_t), st));
    if (B > 0) {
        SPEV_REQUIRE(mel_lens && (T == 0 || (dur && cumsum)), SPEV_E_INVALID, "lr_plan: null buffer");
        const int wpb = 4;
        const int grid = std::min((B + wpb - 1) / wpb, 148 * 8);
        auto ml = reinterpret_cast<long long*>(mel_lens);
        auto mx = reinterpret_cast<long long*>(max_len_dev);
        switch (dur_dtype) {
            case 0: k_lr_plan<<<grid, wpb * 32, 0, st>>>(static_cast<const long long*>(dur), B, T, cumsum, ml, mx); break;
            case 1: k_lr_plan<<<grid, wpb * 32, 0, st>>>(static_cast<const int*>(dur), B, T, cumsum, ml, mx); break;
            case 2: k_lr_plan<<<grid, wpb * 32, 0, st>>>(static_cast<const float*>(dur), B, T, cumsum, ml, mx); break;
            case 3: k_lr_plan<<<grid, wpb * 32, 0, st>>>(static_cast<const double*>(dur), B, T, cumsum, ml, mx); break;
            case 4: k_lr_plan<<<grid, wpb * 32, 0, st>>>(static_cast<const __half*>(dur), B, T, cumsum, ml, mx); break;
            case 5: k_lr_plan<<<grid, wpb * 32, 0, st>>>(static_cast<const __nv_bfloat16*>(dur), B, T, cumsum, ml, mx); break;
            default: SPEV_REQUIRE(false, SPEV_E_INVALID, "lr_plan: unknown dur_dtype %d", dur_dtype);
        }
        SPEV_CUDA(cudaGetLastError());
    }
    if (max_len_host)
        SPEV_CUDA(cudaMemcpyAsync(max_len_host, max_len_dev, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    return SPEV_OK;
}

int spev_lr_expand_fused(const void* x, int64_t row_bytes, const float* feats, int n_feat,
                         const float* clamp_lo_host, const float* clamp_hi_host, const int32_t* cumsum,
                         int B, int T, void* out, float* feats_out, int64_t max_len, void* stream) {
    SPEV_REQUIRE(B >= 0 && T >= 0 && max_len >= 0 && n_feat >= 0 && n_feat <= 16, SPEV_E_INVALID,
                 "lr_expand: bad shape");
    if (B == 0 || max_len == 0) return SPEV_OK;
    SPEV_REQUIRE(B <= 65535, SPEV_E_UNSUPPORTED, "lr_expand: B > 65535");
    SPEV_REQUIRE(T == 0 || cumsum, SPEV_E_INVALID, "lr_expand: cumsum is null");
    SPEV_REQUIRE(!x || (out && row_bytes > 0), SPEV_E_INVALID, "lr_expand: x given but out/row_bytes missing");
    SPEV_REQUIRE(n_feat == 0 || (feats && feats_out), SPEV_E_INVALID, "lr_expand: feats buffers missing");
    ClampParams cp;
    fill_clamp(cp, n_feat, clamp_lo_host, clamp_hi_host);
    dim3 grid(static_cast<unsigned>((max_len + kLrFrames - 1) / kLrFrames), static_cast<unsigned>(B));
    k_lr_expand<<<grid, kLrThreads, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const unsigned char*>(x), row_bytes,
                                                                            feats, n_feat, cp, cumsum, B, T,
                                                                            static_cast<unsigned char*>(out), feats_out, max_len);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

int spev_lr_expand(const void* x, int64_t row_bytes, const int32_t* cumsum, int B, int T, void* out,
                   int64_t max_len, void* stream) {
    SPEV_REQUIRE(x && out, SPEV_E_INVALID, "spev_lr_expand: null x/out");
    return spev_lr_expand_fused(x, row_bytes, nullptr, 0, nullptr, nullptr, cumsum, B, T, out, nullptr, max_len, stream);
}

int spev_variance_fuse(const float* x, const float* feats, int n_feat, const float* clamp_lo_host, const float* clamp_hi_host,
                       const float* conv_w, const float* conv_b, const int32_t* cumsum, int B, int T, int H, float* out,
                       float* feats_out, int64_t max_len, void* stream) {
    SPEV_REQUIRE(B >= 0 && T >= 0 && H > 0 && max_len >= 0 && n_feat >= 0 && n_feat <= kVaMaxFeat, SPEV_E_INVALID,
                 "variance_fuse: bad shape (n_feat <= %d)", kVaMaxFeat);
    if (B == 0 || max_len == 0) return SPEV_OK;
    SPEV_REQUIRE(B <= 65535, SPEV_E_UNSUPPORTED, "variance_fuse: B > 65535");
    SPEV_REQUIRE(x && out && (T == 0 || cumsum) && (n_feat == 0 || (feats && conv_w && conv_b)), SPEV_E_INVALID,
                 "variance_fuse: null buffer");
    ClampParams cp;
    fill_clamp(cp, n_feat, clamp_lo_host, clamp_hi_host);
    dim3 grid(static_cast<unsigned>((max_len + kVaFrames - 1) / kVaFrames), static_cast<unsigned>(B));
    k_variance_fuse<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, feats, n_feat, cp, conv_w, conv_b, cumsum, B, T, H,
                                                                         out, feats_out, max_len);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

int spev_lr_expand_backward(const void* grad_out, int dtype, int H, const float* grad_feats_out, int n_feat,
                            const float* feats, const float* clamp_lo_host, const float* clamp_hi_host,
                            const int32_t* cumsum, int B, int T, int64_t max_len, void* grad_x, float* grad_feats,
                            void* stream) {
    SPEV_REQUIRE(B >= 0 && T >= 0 && max_len >= 0 && H >= 0 && n_feat >= 0 && n_feat <= kMaxFeat, SPEV_E_INVALID,
                 "lr_expand_backward: bad shape");
    if (B == 0 || T == 0) return SPEV_OK;
    SPEV_REQUIRE(cumsum, SPEV_E_INVALID, "lr_expand_backward: cumsum is null");
    SPEV_REQUIRE((grad_out == nullptr) == (grad_x == nullptr), SPEV_E_INVALID, "lr_expand_backward: grad_out/grad_x must come together");
    SPEV_REQUIRE(n_feat == 0 || (grad_feats_out && grad_feats), SPEV_E_INVALID, "lr_expand_backward: curve gradients missing");
    SPEV_REQUIRE(!(clamp_lo_host && clamp_hi_host) || n_feat == 0 || feats, SPEV_E_INVALID,
                 "lr_expand_backward: the clamp mask needs the forward's feats");
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (grad_out && H > 0) {
        const int64_t n = static_cast<int64_t>(B) * T * H;
        const bool f4 = dtype == 0 && H % 4 == 0 && (reinterpret_cast<uintptr_t>(grad_out) & 15) == 0 &&
                        (reinterpret_cast<uintptr_t>(grad_x) & 15) == 0;
        if (f4) {
            k_lr_expand_bwd_f4<<<grid_for(n / 4, 256), 256, 0, st>>>(static_cast<const float4*>(grad_out), H / 4, cumsum, B, T,
                                                                     max_len, static_cast<float4*>(grad_x));
        } else {
            const int grid = grid_for(n, 256);
            switch (dtype) {
                case 0: k_lr_expand_bwd<<<grid, 256, 0, st>>>(static_cast<const float*>(grad_out), H, cumsum, B, T, max_len, static_cast<float*>(grad_x)); break;
                case 1: k_lr_expand_bwd<<<grid, 256, 0, st>>>(static_cast<const double*>(grad_out), H, cumsum, B, T, max_len, static_cast<double*>(grad_x)); break;
                case 2: k_lr_expand_bwd<<<grid, 256, 0, st>>>(static_cast<const __half*>(grad_out), H, cumsum, B, T, max_len, static_cast<__half*>(grad_x)); break;
                case 3: k_lr_expand_bwd<<<grid, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(grad_out), H, cumsum, B, T, max_len, static_cast<__nv_bfloat16*>(grad_x)); break;
                default: SPEV_REQUIRE(false, SPEV_E_INVALID, "lr_expand_backward: dtype must be 0=f32 1=f64 2=f16 3=bf16 (got %d)", dtype);
            }
        }
        SPEV_CUDA(cudaGetLastError());
    }
    if (n_feat > 0) {
        ClampParams cp;
        fill_clamp(cp, n_feat, clamp_lo_host, clamp_hi_host);
        const int64_t n = static_cast<int64_t>(n_feat) * B * T;
        k_lr_curves_bwd<<<grid_for(n, 256), 256, 0, st>>>(grad_feats_out, feats, n_feat, cp, cumsum, B, T, max_len, grad_feats);
        SPEV_CUDA(cudaGetLastError());
    }
    return SPEV_OK;
}

size_t spev_variance_fuse_backward_workspace_bytes(int n_feat, int B, int H, int64_t max_len) {
    if (n_feat < 0 || B < 0 || H < 0 || max_len < 0) return 0;
    const size_t gcv = static_cast<size_t>(n_feat) * B * max_len * sizeof(float);
    const size_t part = static_cast<size_t>(va_bwd_grid(B, max_len)) * H * (3 * n_feat + 1) * sizeof(float);
    return ((gcv + 255) & ~static_cast<size_t>(255)) + part + 256;
}

int spev_variance_fuse_backward(const float* grad_out, const float* feats, int n_feat, const float* clamp_lo_host,
                                const float* clamp_hi_host, const float* conv_w, const int32_t* cumsum, int B, int T,
                                int H, int64_t max_len, float* grad_x, float* grad_feats, float* grad_w, float* grad_b,
                                void* workspace, size_t workspace_bytes, void* stream) {
    SPEV_REQUIRE(B >= 0 && T >= 0 && H > 0 && max_len >= 0 && n_feat >= 0, SPEV_E_INVALID, "variance_fuse_backward: bad shape");
    SPEV_REQUIRE(n_feat <= 5 && H <= 1024, SPEV_E_UNSUPPORTED,
                 "variance_fuse_backward: at most 5 curves and H <= 1024 (got n_feat=%d, H=%d)", n_feat, H);
    if (B == 0 || max_len == 0) return SPEV_OK;
    SPEV_REQUIRE(grad_out && (T == 0 || cumsum), SPEV_E_INVALID, "variance_fuse_backward: null buffer");
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = SPEV_OK;
    if (grad_x && T > 0) {
        rc = spev_lr_expand_backward(grad_out, 0, H, nullptr, 0, nullptr, nullptr, nullptr, cumsum, B, T, max_len, grad_x,
                                     nullptr, stream);
        if (rc) return rc;
    }
    if (n_feat == 0 || !(grad_feats || grad_w || grad_b)) return SPEV_OK;
    SPEV_REQUIRE(feats && conv_w, SPEV_E_INVALID, "variance_fuse_backward: feats / conv_w missing");
    const size_t need = spev_variance_fuse_backward_workspace_bytes(n_feat, B, H, max_len);
    SPEV_REQUIRE(workspace && workspace_bytes >= need, SPEV_E_WORKSPACE,
                 "variance_fuse_backward: workspace too small (%zu < %zu)", workspace_bytes, need);
    uintptr_t base = (reinterpret_cast<uintptr_t>(workspace) + 255) & ~static_cast<uintptr_t>(255);
    float* grad_cv = reinterpret_cast<float*>(base);
    const size_t gcv = static_cast<size_t>(n_feat) * B * max_len * sizeof(float);
    float* partials = reinterpret_cast<float*>(base + ((gcv + 255) & ~static_cast<size_t>(255)));
    ClampParams cp;
    fill_clamp(cp, n_feat, clamp_lo_host, clamp_hi_host);
    const int grid = va_bwd_grid(B, max_len);
    switch (n_feat) {
        case 1: rc = launch_va_bwd<1>(grad_out, feats, cp, conv_w, cumsum, B, T, H, max_len, grad_cv, partials, grid, st); break;
        case 2: rc = launch_va_bwd<2>(grad_out, feats, cp, conv_w, cumsum, B, T, H, max_len, grad_cv, partials, grid, st); break;
        case 3: rc = launch_va_bwd<3>(grad_out, feats, cp, conv_w, cumsum, B, T, H, max_len, grad_cv, partials, grid, st); break;
        case 4: rc = launch_va_bwd<4>(grad_out, feats, cp, conv_w, cumsum, B, T, H, max_len, grad_cv, partials, grid, st); break;
        default: rc = launch_va_bwd<5>(grad_out, feats, cp, conv_w, cumsum, B, T, H, max_len, grad_cv, partials, grid, st); break;
    }
    if (rc) return rc;
    if (grad_w || grad_b) {
        const int n = H * (3 * n_feat + 1);
        k_variance_bwd_reduce<<<(n + 127) / 128, 128, 0, st>>>(partials, grid, H, n_feat, grad_w, grad_b);
        SPEV_CUDA(cudaGetLastError());
    }
    if (grad_feats && T > 0) {
        // the clamp mask is already applied to grad_cv (and padding frames hold 0): plain segment sums
        ClampParams none;
        fill_clamp(none, 0, nullptr, nullptr);
        const int64_t n = static_cast<int64_t>(n_feat) * B * T;
        k_lr_curves_bwd<<<grid_for(n, 256), 256, 0, st>>>(grad_cv, nullptr, n_feat, none, cumsum, B, T, max_len, grad_feats);
        SPEV_CUDA(cudaGetLastError());
    }
    return SPEV_OK;
}

int spev_duration_rule(const float* log_dur, int64_t n, float d_control, int64_t* dur, void* stream) {
    SPEV_REQUIRE(n >= 0, SPEV_E_INVALID, "duration_rule: n < 0");
    if (n == 0) return SPEV_OK;
    SPEV_REQUIRE(log_dur && dur, SPEV_E_INVALID, "duration_rule: null buffer");
    const int grid = static_cast<int>(std::min<int64_t>((n + 255) / 256, 148 * 8));
    k_duration_rule<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(log_dur, n, d_control, reinterpret_cast<long long*>(dur));
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

int spev_bucketize_embed(const float* v, int64_t n, const float* boundaries, int n_boundaries, int right,
                         const float* table, int H, int64_t* idx_out, float* out, int accumulate, void* stream) {
    SPEV_REQUIRE(n >= 0 && n_boundaries >= 0 && n_boundaries <= 12000, SPEV_E_INVALID, "bucketize: bad sizes (n_boundaries <= 12000)");
    if (n == 0) return SPEV_OK;
    SPEV_REQUIRE(v && (n_boundaries == 0 || boundaries), SPEV_E_INVALID, "bucketize: null input");
    SPEV_REQUIRE(!out || (table && H > 0), SPEV_E_INVALID, "bucketize: out given but table/H missing");
    const int wpb = 8;
    const int64_t groups = (n + 31) / 32;
    const int grid = static_cast<int>(std::min<int64_t>((groups + wpb - 1) / wpb, 148 * 8));
    k_bucketize_embed<<<grid, wpb * 32, sizeof(float) * n_boundaries, static_cast<cudaStream_t>(stream)>>>(
        v, n, boundaries, n_boundaries, right, table, H, reinterpret_cast<long long*>(idx_out), out, accumulate);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

}  // extern "C"
