// spev_internal.cuh -- ctx layout, error plumbing and launch helpers shared by the .cu files.
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <vector>

#include "../../include/spev_b200.h"
#include "fft_core.cuh"

namespace spev {

constexpr int kTileFrames = SPEV_TILE_FRAMES;
constexpr int kTileChunks = SPEV_TILE_CHUNKS;
constexpr int kSpecLd = SPEV_SPEC_LD;
constexpr int kWarps = 16;
constexpr int kThreads = kWarps * 32;
constexpr int kStageSamples = (kTileFrames - 1) * kHop + kNfft;   // 8960

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define SPEV_CUDA(call)                                                        \
    do {                                                                       \
        cudaError_t _e = (call);                                               \
        if (_e != cudaSuccess) return ::spev::cuda_fail(_e, #call);            \
    } while (0)

#define SPEV_REQUIRE(cond, code, ...)                                          \
    do {                                                                       \
        if (!(cond)) {                                                         \
            ::spev::set_error(__VA_ARGS__);                                    \
            return (code);                                                     \
        }                                                                      \
    } while (0)

// Mel projection of the fused kernels as a per-warp band list built on the host: warp w owns the nb bands
// hdr[w*nb .. w*nb+nb) (LPT-balanced; unused slots have mel = -1).  A band is a run of float4 weight groups over
// consecutive bins starting at a multiple of 4: hdr = (first group in gw, first bin, group count, mel index).
struct MelProgram {
    int n_mels;
    int nb;              // bands per warp = ceil(n_mels / 16)
    int n_groups;        // float4 groups in gw
    const float4* gw;    // dev [n_groups]
    const int4* hdr;     // dev [16*nb]
};

}  // namespace spev

struct spev_ctx {
    int device, sr, n_fft, hop, win, n_mels;
    int num_sms;          // CTAs the persistent kernels launch (<= num_sms_device; spev_set_sm_limit)
    int num_sms_device;
    float fmin, fmax;
    // host copies
    std::vector<float> h_basis;      // [n_mels*513]
    std::vector<float> h_pinv;       // [513*n_mels]
    std::vector<float> h_window;     // [1024]
    // device constants
    float2* d_tw;        // [32*32] exp(-2 pi i k1 l / 1024)
    float* d_window;     // [1024] periodic Hann
    float2* d_win2048;   // [1024] 0.5 * periodic Hann-2048 as (w[2n], w[2n+1])  (features.cu)
    float2* d_tw2048;    // [512]  exp(-2 pi i k / 2048)
    float* d_basis;      // [n_mels, 513] dense float32 basis (NNLS objective)
    int* d_nnls_rng;     // banded view of the basis for the NNLS screening kernel: [n_mels] (first bin, count) then [513] (first band, last band)
    float* d_basis_pad;  // [n_mels, 520] zero padded (K-major B operand of the mel GEMM)
    float* d_basis_hi;   // tf32-truncated part, same shape
    float* d_basis_lo;   // residual, same shape
    float* d_pinv_t;     // [n_mels, 520]: pinv transposed (pinv_t[m][k] = pinv[k][m])
    float* d_pinv_hi;    // [528, n_mels_pad]: pinv rows (K-major B operand), tf32 hi
    float* d_pinv_lo;    //   residual
    float4* d_prog_w;    // mel program of the fused kernel (MelProgram)
    int4* d_prog_h;
    int prog_gmax;       // most groups any warp runs (diagnostics)
    int prog_nb, prog_groups;
    int band_nnz;        // nnz of the basis (diagnostics)
    int band_max_len;
    void* tma;           // opaque: tensor-map cache (gemm_tc.cu)
    int use_tc;          // mel->magnitude on frame-major input uses the tcgen05 GEMM
};
