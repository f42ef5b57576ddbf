// collate.cu -- GPU-side batching of a resident cache (SURVEY 8(f) row 3): the ragged -> padded
// copies of the reference's collate_fn (/root/reference/spev_real_metrics.py:449-462:
// pad_sequence(..., batch_first=True) over ids, durs, mel and the six per-phone float curves) as
// ONE launch.  Because every item's rows are contiguous in the flat cache, padding item b of an
// array is a contiguous copy of len_b * row_bytes followed by a zero fill: pure HBM byte work,
// 16-byte vectorised when alignment allows, bit-exact for every dtype.
#include <algorithm>
#include "spev_internal.cuh"

namespace spev {

constexpr int kMaxPadArrays = 12;
struct PadParams {
    int n_arrays, B;
    int64_t t_max, p_max;
    const int64_t* frame_off;
    const int64_t* phone_off;
    const int64_t* sel;
    spev_pad_array a[kMaxPadArrays];
};

constexpr int kPadThreads = 256;
constexpr int kPadBytesPerCta = kPadThreads * 16 * 4;   // 16 KB of output per CTA

__global__ void __launch_bounds__(kPadThreads)
k_pad_ragged(PadParams p) {
    const spev_pad_array arr = p.a[blockIdx.z];
    const int b = blockIdx.y;
    const int64_t item = p.sel ? p.sel[b] : b;
    const int64_t* off = arr.per_phone ? p.phone_off : p.frame_off;
    const int64_t lmax = arr.per_phone ? p.p_max : p.t_max;
    const int64_t row = arr.row_bytes;
    const int64_t valid = (off[item + 1] - off[item]) * row;          // bytes to copy
    const int64_t total = lmax * row;                                 // bytes of the padded block
    const unsigned char* src = static_cast<const unsigned char*>(arr.src) + off[item] * row;
    unsigned char* dst = static_cast<unsigned char*>(arr.dst) + static_cast<int64_t>(b) * total;
    const int64_t lo = static_cast<int64_t>(blockIdx.x) * kPadBytesPerCta;
    const int64_t hi = min(total, lo + kPadBytesPerCta);
    if (lo >= total) return;
    const bool vec = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst) | static_cast<uintptr_t>(valid)) & 15) == 0;
    if (vec) {
        for (int64_t i = lo + threadIdx.x * 16; i < hi; i += kPadThreads * 16) {
            uint4 v = make_uint4(0, 0, 0, 0);
            if (i < valid) v = __ldg(reinterpret_cast<const uint4*>(src + i));
            if (i + 16 <= total) *reinterpret_cast<uint4*>(dst + i) = v;
            else for (int64_t j = i; j < total; ++j) dst[j] = j < valid ? src[j] : 0;
        }
    } else if (((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst) | static_cast<uintptr_t>(row)) & 3) == 0) {
        for (int64_t i = lo + threadIdx.x * 4; i < hi; i += kPadThreads * 4)
            *reinterpret_cast<uint32_t*>(dst + i) = i < valid ? __ldg(reinterpret_cast<const uint32_t*>(src + i)) : 0u;
    } else {
        for (int64_t i = lo + threadIdx.x; i < hi; i += kPadThreads) dst[i] = i < valid ? src[i] : 0;
    }
}

// ---- segmented copy: dst[dst_off[i] .. +nbytes[i]) = src[src_off[i] .. +nbytes[i]) -------------------------------
// Re-orders a gathered cache (rank-major rows) into corpus order, or packs scattered utterances into a shard: each
// segment is a contiguous run of rows.  CTA <-> 16 KB piece of one segment (binary search in the piece prefix table).
__global__ void __launch_bounds__(kPadThreads)
k_copy_segments(const unsigned char* __restrict__ src, unsigned char* __restrict__ dst, const int64_t* __restrict__ src_off,
                const int64_t* __restrict__ dst_off, const int64_t* __restrict__ nbytes, const int64_t* __restrict__ piece_off,
                int n_seg, int64_t n_pieces) {
    for (int64_t piece = blockIdx.x; piece < n_pieces; piece += gridDim.x) {
        int lo = 0, hi = n_seg;                       // last segment whose first piece is <= piece
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (piece_off[mid] <= piece) lo = mid; else hi = mid;
        }
        const int64_t b0 = (piece - piece_off[lo]) * kPadBytesPerCta;
        const int64_t b1 = min(nbytes[lo], b0 + kPadBytesPerCta);
        const unsigned char* s = src + src_off[lo];
        unsigned char* d = dst + dst_off[lo];
        if (((reinterpret_cast<uintptr_t>(s) | reinterpret_cast<uintptr_t>(d)) & 15) == 0) {
            const int64_t v1 = b0 + ((b1 - b0) & ~static_cast<int64_t>(15));
            for (int64_t i = b0 + threadIdx.x * 16; i < v1; i += kPadThreads * 16)
                *reinterpret_cast<uint4*>(d + i) = __ldg(reinterpret_cast<const uint4*>(s + i));
            for (int64_t i = v1 + threadIdx.x; i < b1; i += kPadThreads) d[i] = s[i];
        } else if (((reinterpret_cast<uintptr_t>(s) | reinterpret_cast<uintptr_t>(d) | static_cast<uintptr_t>(b1 - b0)) & 3) == 0) {
            for (int64_t i = b0 + threadIdx.x * 4; i < b1; i += kPadThreads * 4)
                *reinterpret_cast<uint32_t*>(d + i) = __ldg(reinterpret_cast<const uint32_t*>(s + i));
        } else {
            for (int64_t i = b0 + threadIdx.x; i < b1; i += kPadThreads) d[i] = s[i];
        }
    }
}

// ---- batched 2-D transpose: dst[b][c][r] = src[b][r][c] -------------------------------------------------------------
// librosa lays spectra and mels out as [..., bins, T]; the kernels here work on frame-major rows [F, pitch].  This is
// the layout change between the two (32 x 32 tiles through padded shared memory, coalesced on both sides), for 4-byte
// (float) and 8-byte (complex64) elements, with independent row pitches and batch strides on either side so that the
// 520-column padded spectra are read / written in place.
template <class T>
__global__ void __launch_bounds__(256)
k_transpose(const T* __restrict__ src, T* __restrict__ dst, int rows, int cols, int64_t src_pitch, int64_t src_batch,
            int64_t dst_pitch, int64_t dst_batch) {
    __shared__ T tile[32][33];
    const int64_t b = blockIdx.z;
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;        // 32 x 8
    const T* s = src + b * src_batch;
    T* d = dst + b * dst_batch;
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
        const int r = r0 + ty + j, c = c0 + tx;
        if (r < rows && c < cols) tile[ty + j][tx] = s[static_cast<int64_t>(r) * src_pitch + c];
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
        const int c = c0 + ty + j, r = r0 + tx;
        if (r < rows && c < cols) d[static_cast<int64_t>(c) * dst_pitch + r] = tile[tx][ty + j];
    }
}

}  // namespace spev

using namespace spev;

extern "C" {

int spev_collate(const spev_pad_array* arrays, int n_arrays, const int64_t* frame_off, const int64_t* phone_off,
                 const int64_t* sel, int B, int64_t t_max, int64_t p_max, void* stream) {
    SPEV_REQUIRE(n_arrays >= 0 && n_arrays <= kMaxPadArrays && B >= 0 && t_max >= 0 && p_max >= 0, SPEV_E_INVALID,
                 "collate: bad sizes (at most %d arrays)", kMaxPadArrays);
    if (n_arrays == 0 || B == 0) return SPEV_OK;
    SPEV_REQUIRE(arrays && B <= 65535, SPEV_E_INVALID, "collate: null arrays or B > 65535");
    PadParams p{};
    p.n_arrays = n_arrays; p.B = B; p.t_max = t_max; p.p_max = p_max;
    p.frame_off = frame_off; p.phone_off = phone_off; p.sel = sel;
    int64_t max_bytes = 0;
    for (int i = 0; i < n_arrays; ++i) {
        SPEV_REQUIRE(arrays[i].src && arrays[i].dst && arrays[i].row_bytes > 0, SPEV_E_INVALID, "collate: array %d incomplete", i);
        SPEV_REQUIRE(arrays[i].per_phone ? phone_off != nullptr : frame_off != nullptr, SPEV_E_INVALID,
                     "collate: array %d needs an offset table that was not given", i);
        p.a[i] = arrays[i];
        max_bytes = std::max(max_bytes, (arrays[i].per_phone ? p_max : t_max) * arrays[i].row_bytes);
    }
    if (max_bytes == 0) return SPEV_OK;
    dim3 grid(static_cast<unsigned>((max_bytes + kPadBytesPerCta - 1) / kPadBytesPerCta), static_cast<unsigned>(B),
              static_cast<unsigned>(n_arrays));
    k_pad_ragged<<<grid, kPadThreads, 0, static_cast<cudaStream_t>(stream)>>>(p);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

int spev_transpose_batched(const void* src, void* dst, int elem_bytes, int64_t batches, int rows, int cols, int64_t src_pitch,
                           int64_t src_batch, int64_t dst_pitch, int64_t dst_batch, void* stream) {
    SPEV_REQUIRE(batches >= 0 && rows >= 0 && cols >= 0, SPEV_E_INVALID, "transpose: negative shape");
    if (batches == 0 || rows == 0 || cols == 0) return SPEV_OK;
    SPEV_REQUIRE(src && dst && src_pitch >= cols && dst_pitch >= rows, SPEV_E_INVALID, "transpose: null buffer or pitch < extent");
    SPEV_REQUIRE(elem_bytes == 4 || elem_bytes == 8, SPEV_E_UNSUPPORTED, "transpose: 4- or 8-byte elements only");
    SPEV_REQUIRE(batches <= 65535, SPEV_E_UNSUPPORTED, "transpose: more than 65535 batches");
    dim3 grid(static_cast<unsigned>((cols + 31) / 32), static_cast<unsigned>((rows + 31) / 32), static_cast<unsigned>(batches));
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (elem_bytes == 4)
        k_transpose<float><<<grid, 256, 0, st>>>(static_cast<const float*>(src), static_cast<float*>(dst), rows, cols, src_pitch,
                                                src_batch, dst_pitch, dst_batch);
    else
        k_transpose<float2><<<grid, 256, 0, st>>>(static_cast<const float2*>(src), static_cast<float2*>(dst), rows, cols, src_pitch,
                                                 src_batch, dst_pitch, dst_batch);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

int spev_copy_segments_piece_bytes(void) { return kPadBytesPerCta; }

int spev_copy_segments(const void* src, void* dst, const int64_t* src_off, const int64_t* dst_off, const int64_t* nbytes,
                       const int64_t* piece_off, int n_seg, int64_t n_pieces, void* stream) {
    SPEV_REQUIRE(n_seg >= 0 && n_pieces >= 0, SPEV_E_INVALID, "copy_segments: negative sizes");
    if (n_seg == 0 || n_pieces == 0) return SPEV_OK;
    SPEV_REQUIRE(src && dst && src_off && dst_off && nbytes && piece_off, SPEV_E_INVALID, "copy_segments: null buffer");
    const int grid = static_cast<int>(std::min<int64_t>(n_pieces, 148 * 32));
    k_copy_segments<<<grid, kPadThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const unsigned char*>(src), static_cast<unsigned char*>(dst), src_off, dst_off, nbytes, piece_off, n_seg, n_pieces);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

}  // extern "C"
