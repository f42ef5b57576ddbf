// gemm_tc.cu -- TMA-staged tcgen05 GEMM engine (3xTF32) for the mel projection and its
// pseudo-inverse:     D[M, N] = A[M, K] . B[N, K]^T      (fp32 in, fp32 out)
//
//   K2  spev_mel_project : power[F, 513(520)] . basis[80, 513]^T -> log/clamp -> [F, 80]
//       replaces the einsum inside librosa.feature.melspectrogram + :364-366
//       (/root/reference/spev_real_metrics.py:363-366)
//   K3' mel_to_mag (TC)  : exp(logmel)[F, 80] . pinv[513, 80]^T -> clip, sqrt -> S[F, 513(520)]
//       replaces librosa.feature.inverse.mel_to_stft under :730
//
// One CTA = MT 128 x BN output tiles, 10 warps, warp-specialised:
//   warp 0      TMA producer: cp.async.bulk.tensor (SWIZZLE_128B, K-major, 32-float K chunks) of
//               the A tiles into a ring of three LANDING buffers and of the pre-split B_hi / B_lo
//               chunks into a 2-slot ring (mbarrier complete_tx).
//   warps 2..9  splitter: 3xTF32 needs A = A_hi + A_lo with A_hi exactly representable in TF32.
//               kind::tf32 ignores the low 13 mantissa bits of its operands, so the tile as it
//               landed IS A_hi and is left alone (with a fused exp() it is rewritten); the splitter
//               writes A_lo = A - (bits & 0xFFFFE000) into ONE shared residual tile -- elementwise,
//               so the swizzled placement is preserved without knowing it -- then fence.proxy.async
//               and arrive on "lo_full".  Later the same warps run the epilogue.
//   warp 1      TMEM allocator + MMA issuer: one elected thread issues, per 8-wide K step,
//               tcgen05.mma.kind::tf32  D += A.B_lo ; D += A.B_hi  as soon as the tile has landed, and
//               D += A_lo.B_hi once the residual is ready, with the accumulators in TMEM (fp32,
//               128 lanes x MT*BN columns); tcgen05.commit -> "empty_a" (landing buffer) and
//               "lo_empty" (residual tile), finally "tmem_full".
//   epilogue    tcgen05.ld 32x32b.x16 (warp w owns TMEM lanes 32*(w%4)..), log/clamp or
//               clip/sqrt in registers, 16-byte row stores.
// Every mbarrier wait is bounded: a protocol bug traps instead of hanging the GPU.
#include <cuda.h>
#include <algorithm>
#include <cstring>
#include "spev_internal.cuh"

namespace spev {

#ifndef SPEV_TC_NSA
#define SPEV_TC_NSA 3
#endif
#ifndef SPEV_TC_NLO
#define SPEV_TC_NLO 1
#endif
#ifndef SPEV_TC_CTAS
#define SPEV_TC_CTAS 2
#endif
constexpr int kBM = 128, kBK = 32;
constexpr int kTcSplit = 256;                  // splitter / epilogue threads (8 warps)
constexpr int kTcThreads = 64 + kTcSplit;
constexpr uint32_t kABytes = kBM * kBK * 4;   // 16 KB

enum { EPI_MEL = 0, EPI_MAG = 1 };

struct TcParams {
    int m_total;        // rows of A / D
    int k_chunks;       // ceil(K / 32)
    int n_valid;        // valid output columns (80 / 513)
    int64_t ld_out;     // row pitch of the output, elements
    int a_exp;          // apply exp() to A before the split
    int log_mode;       // EPI_MEL: 1 -> clamp(log(max(x, floor)), lo, hi)
    float floor_v, lo, hi;
};

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0;
    for (uint32_t spin = 0; !done; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done) : "r"(addr), "r"(parity) : "memory");
        if (spin > (1u << 26)) asm volatile("trap;\n");   // bounded: never hang the device
    }
}
__device__ __forceinline__ void tma_load_2d(void* smem, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n"
        ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
//   [0,14) start>>4 | [16,30) LBO>>4 (unused for swizzled K-major) | [32,46) SBO>>4 = 1024>>4 |
//   [46,48) version = 1 | [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    return static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// cute::UMMA::InstrDescriptor: c=F32 (1<<4), a=b=TF32 (2<<7, 2<<10), K-major both, N>>3 @17, M>>4 @24
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int m, int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}

// One CTA owns MT consecutive 128-row tiles of A and keeps their MT accumulators side by side in TMEM.  The K loop
// runs over (k-chunk, tile) pairs: a chunk of the pre-split B operand (hi + lo) is loaded ONCE per k-chunk into its
// own 2-slot ring and used by all MT tiles, while the A tiles stream through a ring of their own.  With MT = 1 every
// CTA re-reads the whole B operand (333 KB for the mel basis) from L2 per 128 rows -- more bytes than the A tile it
// multiplies (266 KB), and the L2 -> SM path, not HBM, was the limiter (r01: 49 % of the HBM roofline, tensor pipe
// 31 %); MT = 3 cuts the B traffic to a third.
template <int BN, int MT>
struct TcSmem {
    static constexpr int kStagesA = BN > 128 ? 3 : SPEV_TC_NSA;                 // A ring of LANDING buffers; the tf32 residual tile is one shared buffer
    static constexpr int kLo = SPEV_TC_NLO;            // residual (A_lo) tiles
    static constexpr int kSlotsB = 2;                  // B ring (per slot: B_hi + B_lo chunk)
    static constexpr int kCtas = BN > 128 ? 1 : SPEV_TC_CTAS;     // two CTAs per SM: one's epilogue overlaps the other's main loop
    static constexpr uint32_t kBBytes = BN * kBK * 4;
    static constexpr uint32_t kStageA = kABytes;
    static constexpr uint32_t kSlotB = 2 * kBBytes;
    static constexpr uint32_t kBars = 1024;
    static constexpr uint32_t kTotal = kStagesA * kStageA + kLo * kABytes /*A_lo*/ + kSlotsB * kSlotB + kBars + 1024 /*alignment slack*/;
    static constexpr uint32_t kCols = BN * MT;
    static constexpr uint32_t kTmemCols = kCols <= 32 ? 32 : kCols <= 64 ? 64 : kCols <= 128 ? 128 : kCols <= 256 ? 256 : 512;
    static_assert(kCols <= 512 && kTmemCols * kCtas <= 512, "accumulators do not fit TMEM");
};

template <int BN, int EPI, int MT>
__global__ void __launch_bounds__(kTcThreads, TcSmem<BN, MT>::kCtas)
k_gemm_tf32x3(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_bhi,
              const __grid_constant__ CUtensorMap map_blo, float* __restrict__ out, TcParams p) {
    using L = TcSmem<BN, MT>;
    constexpr int NSA = L::kStagesA, NSB = L::kSlotsB;
    extern __shared__ unsigned char smem_raw[];
    // 1024-byte alignment by POINTER arithmetic on the shared-memory symbol: the address space stays known to the compiler
    // (LDS / STS in the splitter; the integer round trip made them generic LD / ST with long-scoreboard latency)
    unsigned char* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* base_lo = base + NSA * L::kStageA;          // the one A_lo tile
    constexpr int NLO = L::kLo;
    unsigned char* base_b = base_lo + NLO * kABytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(base_b + NSB * L::kSlotB);
    uint64_t* full_a = bars;                        // [NSA] TMA landed an A tile
    uint64_t* empty_a = full_a + NSA;               // [NSA] MMAs (and the splitter) done reading the landing buffer
    uint64_t* lo_full = empty_a + NSA;              // [NLO] A_lo written (and, with a_exp, the landing buffer rewritten)
    uint64_t* lo_empty = lo_full + NLO;             // [NLO] the A_lo MMAs of an earlier tile are done with the residual tile
    uint64_t* full_b = lo_empty + NLO;              // [NSB] TMA landed a B chunk
    uint64_t* empty_b = full_b + NSB;               // [NSB] MMAs of every tile done reading the B chunk
    uint64_t* tmem_full = empty_b + NSB;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(tmem_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * (kBM * MT), n0 = blockIdx.y * BN;

    if (threadIdx.x == 0) {
        // a landing buffer is free once its hi products are done (commit: 1) AND every splitter thread has read it
        for (int s = 0; s < NSA; ++s) { mbar_init(full_a + s, 1); mbar_init(empty_a + s, 1 + kTcSplit); }
        for (int q = 0; q < NLO; ++q) { mbar_init(lo_full + q, kTcSplit); mbar_init(lo_empty + q, 1); }
        for (int s = 0; s < NSB; ++s) { mbar_init(full_b + s, 1); mbar_init(empty_b + s, 1); }
        mbar_init(tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(s_tmem)), "n"(L::kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;

    if (warp == 0) {
        if (lane == 0) {
            for (int kc = 0; kc < p.k_chunks; ++kc) {
                const int sb = kc % NSB;
                mbar_wait(empty_b + sb, ((kc / NSB) & 1) ^ 1);
                unsigned char* bs = base_b + sb * L::kSlotB;
                mbar_expect_tx(full_b + sb, 2 * L::kBBytes);
                tma_load_2d(bs, &map_bhi, full_b + sb, kc * kBK, n0);
                tma_load_2d(bs + L::kBBytes, &map_blo, full_b + sb, kc * kBK, n0);
#pragma unroll 1
                for (int mt = 0; mt < MT; ++mt) {
                    const int j = kc * MT + mt, s = j % NSA;
                    mbar_wait(empty_a + s, ((j / NSA) & 1) ^ 1);
                    mbar_expect_tx(full_a + s, kABytes);
                    tma_load_2d(base + s * L::kStageA, &map_a, full_a + s, kc * kBK, m0 + mt * kBM);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_tf32(kBM, BN);
            for (int kc = 0; kc < p.k_chunks; ++kc) {
                const int sb = kc % NSB;
                mbar_wait(full_b + sb, (kc / NSB) & 1);
                const uint32_t b_hi = smem_u32(base_b + sb * L::kSlotB), b_lo = b_hi + L::kBBytes;
#pragma unroll 1
                for (int mt = 0; mt < MT; ++mt) {
                    const int j = kc * MT + mt, s = j % NSA;
                    const int ql = j % NLO;
                    const uint32_t a_hi = smem_u32(base + s * L::kStageA), a_lo = smem_u32(base_lo + ql * kABytes);
                    const uint32_t acc = tmem_base + static_cast<uint32_t>(mt * BN);
                    // kind::tf32 ignores the low 13 mantissa bits of its operands: the tile as it landed IS A_hi, so its
                    // two products start while the splitter is still computing the residual (with a_exp the splitter
                    // rewrites the tile first)
                    auto mma_hi = [&]() {
#pragma unroll
                        for (int k = 0; k < kBK / 8; ++k) {   // UMMA_K = 8 for tf32 = 32 bytes along the swizzled row
                            const uint32_t off = k * 32;
                            const uint64_t dah = umma_desc_sw128(a_hi + off);
                            tc_mma_tf32(acc, dah, umma_desc_sw128(b_lo + off), idesc, (kc | k) != 0);   // small term first
                            tc_mma_tf32(acc, dah, umma_desc_sw128(b_hi + off), idesc, 1);
                        }
                    };
                    mbar_wait(full_a + s, (j / NSA) & 1);
                    tc_fence_after();
                    if (!p.a_exp) { mma_hi(); tc_commit(empty_a + s); }   // (commit implies tcgen05.fence::before_thread_sync)
                    mbar_wait(lo_full + ql, (j / NLO) & 1);
                    tc_fence_after();
                    if (p.a_exp) { mma_hi(); tc_commit(empty_a + s); }
#pragma unroll
                    for (int k = 0; k < kBK / 8; ++k) {
                        const uint32_t off = k * 32;
                        tc_mma_tf32(acc, umma_desc_sw128(a_lo + off), umma_desc_sw128(b_hi + off), idesc, 1);
                    }
                    tc_commit(lo_empty + ql);
                }
                tc_commit(empty_b + sb);
            }
            tc_commit(tmem_full);
        }
    } else {
        const int t = threadIdx.x - 64;   // 0..kTcSplit-1
        const int n_it = p.k_chunks * MT;
        for (int j = 0; j < n_it; ++j) {
            const int s = j % NSA;
            mbar_wait(full_a + s, (j / NSA) & 1);
            float4* a = reinterpret_cast<float4*>(base + s * L::kStageA);
            const int ql = j % NLO;
            float4* l = reinterpret_cast<float4*>(base_lo + ql * kABytes);
            constexpr int kPer = static_cast<int>(kABytes / 16 / kTcSplit);
            float4 lo[kPer];
            // the residuals are computed in registers BEFORE waiting for the residual tile: the loads and the arithmetic
            // overlap the previous tile's A_lo products
#pragma unroll
            for (int i = 0; i < kPer; ++i) {
                float4 v = a[t + kTcSplit * i];
                if (p.a_exp) { v.x = expf(v.x); v.y = expf(v.y); v.z = expf(v.z); v.w = expf(v.w); }
                float4 h;
                h.x = __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
                h.y = __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
                h.z = __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
                h.w = __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
                if (p.a_exp) a[t + kTcSplit * i] = h;       // only exp() changes what the tensor core must see
                lo[i] = make_float4(v.x - h.x, v.y - h.y, v.z - h.z, v.w - h.w);
            }
            if (!p.a_exp) mbar_arrive(empty_a + s);    // this thread is done with the landing buffer
            mbar_wait(lo_empty + ql, ((j / NLO) & 1) ^ 1);   // an earlier tile's A_lo products are done with the residual tile
#pragma unroll
            for (int i = 0; i < kPer; ++i) l[t + kTcSplit * i] = lo[i];
            asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // generic writes -> async proxy (UMMA)
            if (p.a_exp) mbar_arrive(empty_a + s);     // (rewritten tile: counted once its writes are fenced)
            mbar_arrive(lo_full + ql);
        }
        // ---------------- epilogue: TMEM -> registers -> global ----------------
        mbar_wait(tmem_full, 0);
        tc_fence_after();
        const int q = warp & 3;                       // TMEM lane quarter this warp may access
#pragma unroll 1
        for (int mt = 0; mt < MT; ++mt) {
            const int row = m0 + mt * kBM + q * 32 + lane;
            const bool row_ok = row < p.m_total;
            float* orow = out + static_cast<int64_t>(row) * p.ld_out + n0;
#pragma unroll 1
            for (int c0 = ((warp - 2) >> 2) * 16; c0 < BN; c0 += 16 * (kTcSplit / 128)) {   // warps 2..5 / 6..9: alternate 16-column groups
                uint32_t r[16];
                tc_ld16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(mt * BN + c0), r);
                float v[16];
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) {
                    float x = __uint_as_float(r[jj]);
                    if (EPI == EPI_MEL) {
                        if (p.log_mode) x = fminf(fmaxf(logf(fmaxf(x, p.floor_v)), p.lo), p.hi);
                    } else {
                        x = sqrtf(fmaxf(x, 0.f));
                    }
                    v[jj] = x;
                }
                if (row_ok) {
#pragma unroll
                    for (int jj = 0; jj < 16; jj += 4)
                        if (n0 + c0 + jj < p.n_valid)   // n_valid is a multiple of 4 (80 / 520)
                            *reinterpret_cast<float4*>(orow + c0 + jj) = make_float4(v[jj], v[jj + 1], v[jj + 2], v[jj + 3]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(L::kTmemCols) : "memory");
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct TcState {
    EncodeTiledFn encode = nullptr;
    CUtensorMap mel_bhi, mel_blo, pinv_bhi, pinv_blo;
};

// 2-D fp32 row-major tensor [rows, cols] (row pitch `pitch_elems`), box = [box_rows, 32 floats],
// 128-byte swizzle, out-of-bounds elements read as zero.
static int encode_2d(TcState* st, CUtensorMap* map, const float* ptr, uint64_t rows, uint64_t cols,
                     uint64_t pitch_elems, uint32_t box_rows) {
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {pitch_elems * sizeof(float)};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(kBK), box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = st->encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SPEV_REQUIRE(r == CUDA_SUCCESS, SPEV_E_CUDA, "cuTensorMapEncodeTiled failed (CUresult %d)", static_cast<int>(r));
    return SPEV_OK;
}

static float tf32_hi(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    u &= 0xFFFFE000u;
    memcpy(&x, &u, 4);
    return x;
}

// The tf32 hi / residual splits of both B operands: the mel basis zero padded to [n_mels, 520] and pinv [513, n_mels].
int gemm_tc_init(spev_ctx* c) {
    TcState* st = new TcState();
    c->tma = st;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    SPEV_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    SPEV_REQUIRE(fn && qres == cudaDriverEntryPointSuccess, SPEV_E_CUDA, "cuTensorMapEncodeTiled not available");
    st->encode = reinterpret_cast<EncodeTiledFn>(fn);
    const int nm = c->n_mels;
    std::vector<float> b_hi(static_cast<size_t>(nm) * kSpecLd, 0.f), b_lo(b_hi.size(), 0.f);
    for (int m = 0; m < nm; ++m)
        for (int k = 0; k < kBins; ++k) {
            const float v = c->h_basis[static_cast<size_t>(m) * kBins + k];
            const size_t i = static_cast<size_t>(m) * kSpecLd + k;
            b_hi[i] = tf32_hi(v); b_lo[i] = v - b_hi[i];
        }
    std::vector<float> p_hi(c->h_pinv.size()), p_lo(c->h_pinv.size());
    for (size_t i = 0; i < p_hi.size(); ++i) { p_hi[i] = tf32_hi(c->h_pinv[i]); p_lo[i] = c->h_pinv[i] - p_hi[i]; }
    int rc;
    if ((rc = upload(&c->d_basis_hi, b_hi)) || (rc = upload(&c->d_basis_lo, b_lo)) || (rc = upload(&c->d_pinv_hi, p_hi)) ||
        (rc = upload(&c->d_pinv_lo, p_lo)))
        return rc;
    SPEV_CUDA(cudaFuncSetAttribute(k_gemm_tf32x3<80, EPI_MEL, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(TcSmem<80, 3>::kTotal)));
    SPEV_CUDA(cudaFuncSetAttribute(k_gemm_tf32x3<176, EPI_MAG, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(TcSmem<176, 1>::kTotal)));
    if (nm % 4 != 0) return SPEV_OK;   // TMA needs 16-byte row pitches; the TC path is then unavailable
    if ((rc = encode_2d(st, &st->mel_bhi, c->d_basis_hi, nm, kBins, kSpecLd, 80))) return rc;
    if ((rc = encode_2d(st, &st->mel_blo, c->d_basis_lo, nm, kBins, kSpecLd, 80))) return rc;
    if ((rc = encode_2d(st, &st->pinv_bhi, c->d_pinv_hi, kBins, nm, nm, 176))) return rc;
    if ((rc = encode_2d(st, &st->pinv_blo, c->d_pinv_lo, kBins, nm, nm, 176))) return rc;
    return SPEV_OK;
}

void gemm_tc_destroy(spev_ctx* c) {
    delete static_cast<TcState*>(c->tma);
    c->tma = nullptr;
}

template <int BN, int EPI, int MT>
static int launch_tc(const CUtensorMap& ma, const CUtensorMap& mbh, const CUtensorMap& mbl, float* out, const TcParams& p,
                     int n_tiles, cudaStream_t st) {
    auto kern = k_gemm_tf32x3<BN, EPI, MT>;
    using L = TcSmem<BN, MT>;
    dim3 grid(static_cast<unsigned>((p.m_total + kBM * MT - 1) / (kBM * MT)), static_cast<unsigned>(n_tiles));
    kern<<<grid, kTcThreads, L::kTotal, st>>>(ma, mbh, mbl, out, p);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

// mel [F, n_mels] frame-major (layout 0) -> S [F, ld_s]
int mel_to_mag_tc(spev_ctx* c, const float* mel, int64_t n_frames, int is_log, float* S, int64_t ld_s, cudaStream_t stm) {
    TcState* st = static_cast<TcState*>(c->tma);
    SPEV_REQUIRE(st && st->encode, SPEV_E_UNSUPPORTED, "tensor-core path unavailable");
    SPEV_REQUIRE(n_frames < (1ll << 31), SPEV_E_INVALID, "mel_to_mag (tc): need ld_s >= 520, multiple of 4");
    CUtensorMap ma;
    int rc = encode_2d(st, &ma, mel, static_cast<uint64_t>(n_frames), c->n_mels, c->n_mels, kBM);
    if (rc) return rc;
    TcParams p{};
    p.m_total = static_cast<int>(n_frames); p.k_chunks = (c->n_mels + kBK - 1) / kBK; p.n_valid = kSpecLd; p.ld_out = ld_s;
    p.a_exp = is_log; p.log_mode = 0;
    return launch_tc<176, EPI_MAG, 1>(ma, st->pinv_bhi, st->pinv_blo, S, p, 3, stm);
}

}  // namespace spev

using namespace spev;

extern "C" {

int spev_mel_project(spev_ctx* c, const float* power, int64_t n_frames, float* out, int mode, float floor_v, float lo,
                     float hi, void* stream) {
    SPEV_ON_CTX_DEVICE(c);
    SPEV_REQUIRE(mode == 0 || mode == 1, SPEV_E_INVALID, "spev_mel_project: mode must be 0 or 1");
    TcState* st = static_cast<TcState*>(c->tma);
    SPEV_REQUIRE(st && st->encode, SPEV_E_UNSUPPORTED, "tensor-core path unavailable");
    SPEV_REQUIRE(c->n_mels == 80, SPEV_E_UNSUPPORTED, "spev_mel_project: tensor-core path is built for n_mels=80");
    SPEV_REQUIRE(n_frames >= 0 && n_frames < (1ll << 31), SPEV_E_INVALID, "spev_mel_project: bad n_frames");
    if (n_frames == 0) return SPEV_OK;
    SPEV_REQUIRE(power && out && (reinterpret_cast<uintptr_t>(power) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                 SPEV_E_INVALID, "spev_mel_project: null or unaligned buffer");
    CUtensorMap ma;
    int rc = encode_2d(st, &ma, power, static_cast<uint64_t>(n_frames), kBins, kSpecLd, kBM);
    if (rc) return rc;
    TcParams p{};
    p.m_total = static_cast<int>(n_frames); p.k_chunks = (kBins + kBK - 1) / kBK; p.n_valid = 80; p.ld_out = 80;
    p.a_exp = 0; p.log_mode = mode; p.floor_v = floor_v; p.lo = lo; p.hi = hi;
    return launch_tc<80, EPI_MEL, 3>(ma, st->mel_bhi, st->mel_blo, out, p, 1, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
