// spev_internal.cuh -- ctx layout, error plumbing and launch helpers shared by the .cu files.
#pragma once
#include <cuda_runtime.h>
#include <algorithm>
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
    float* d_window;     // [1024] periodic Hann, then [256] 1 / window-sum-square of interior ISTFT chunks
    float2* d_win2048;   // [1024] 0.5 * periodic Hann-2048 as (w[2n], w[2n+1])  (features.cu)
    float2* d_tw2048;    // [512]  exp(-2 pi i k / 2048)
    float* d_basis;      // [n_mels, 513] dense float32 basis (NNLS objective)
    int* d_nnls_rng;     // banded view of the basis for the NNLS screening kernel: [n_mels] (first bin, count) then [513] (first band, last band)
    float* d_basis_hi;   // [n_mels, 520] zero padded basis (K-major B operand of the mel GEMM), tf32 hi
    float* d_basis_lo;   //   residual
    float* d_pinv_t;     // [n_mels, 520]: pinv transposed (pinv_t[m][k] = pinv[k][m])
    float* d_pinv_hi;    // [513, n_mels]: pinv rows (K-major B operand of the mel->magnitude GEMM), tf32 hi
    float* d_pinv_lo;    //   residual
    float4* d_prog_w;    // mel program of the fused kernel (MelProgram, spectral.cu)
    int4* d_prog_h;
    int prog_nb, prog_groups;
    void* tma;           // opaque: tensor-map cache (gemm_tc.cu)
    int use_tc;          // mel->magnitude on frame-major input uses the tcgen05 GEMM
};

namespace spev {

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
    ::spev::DeviceGuard _guard(c); \
    if (_guard.rc) return _guard.rc

// Copy a host table to a new device allocation (at least one element, so an empty table still gets a valid pointer).
template <class T>
int upload(T** dst, const std::vector<T>& src) {
    SPEV_CUDA(cudaMalloc(reinterpret_cast<void**>(dst), std::max<size_t>(1, src.size()) * sizeof(T)));
    if (!src.empty())
        SPEV_CUDA(cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
    return SPEV_OK;
}

// Per-file parts of spev_create: each builds and uploads the ctx tables only its own kernels read, from h_basis,
// h_pinv and h_window.  spev_destroy frees them.
int spectral_init(spev_ctx* c);
int gemm_tc_init(spev_ctx* c);
void gemm_tc_destroy(spev_ctx* c);
int nnls_init(spev_ctx* c);
int features_init(spev_ctx* c);

// spev_mel_to_mag on frame-major input (gemm_tc.cu).  The caller has checked n_mels % 4 == 0, n_frames > 0,
// ld_s >= 520 with ld_s % 4 == 0, and 16-byte aligned mel and S.
int mel_to_mag_tc(spev_ctx* c, const float* mel, int64_t n_frames, int is_log, float* S, int64_t ld_s, cudaStream_t st);

}  // namespace spev
