// nnls.cu -- objective / gradient of librosa.util.nnls for the mel -> linear inversion.
//
// librosa.feature.inverse.mel_to_stft (reached from /root/reference/spev_real_metrics.py:730-733) solves
//     min_x>=0  f(x) = (0.5 / B.size) * || A x - B ||^2        A = mel basis [n_mels, 513],  B = a block of mel columns
// with scipy's L-BFGS-B started at x0 = clip(pinv(A) B, 0), block by block (MAX_MEM_BLOCK columns at a time).  For
// reference-range inputs and blocks of >~ 40 columns the projected gradient at x0 is already below pgtol and x0 is
// returned; short utterances and short remainder blocks do iterate (up to ~50 % change, DESIGN.md "NNLS").
// This kernel evaluates f, its gradient (1 / B.size) A^T (A x - B) and the projected-gradient sup-norm of L-BFGS-B's
// convergence test in float64 -- the precision librosa's objective runs in (scipy hands it a float64 x) -- one CTA
// per column.  The optimizer's control flow stays on the host (scipy, exactly the routine librosa calls).
#include "spev_internal.cuh"

namespace spev {

constexpr int kNnlsThreads = 256;

// XMODE 0: x float64 in librosa's order [L, 513, tb];  1: x = S^2 from float32 magnitude rows S (row = l*T + t0 + t,
// pitch ld_x) -- the warm start clip(pinv B, 0) as spev_mel_to_mag leaves it (its square root)
// Real = double: librosa's precision (every call that feeds L-BFGS-B).  Real = float: the screening pass over all blocks
// of a call -- it only has to decide "projected gradient above or below pgtol", and blocks it finds within 10 % of the
// threshold are re-evaluated in double by the caller.
template <int XMODE, class Real>
__global__ void __launch_bounds__(kNnlsThreads)
k_nnls_objective(const void* __restrict__ xv, int64_t ld_x, const float* __restrict__ mel /*[L*T, n_mels]*/, int is_log,
                 const float* __restrict__ basis /*[n_mels, 513]*/, int n_mels, int L, int64_t T, int64_t t0, int tb,
                 double inv_size, double* __restrict__ value_parts, double* __restrict__ grad /*[L,513,tb] or null*/,
                 double* __restrict__ pg_max) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Real* s_x = reinterpret_cast<Real*>(smem_raw);           // [513]
    Real* s_r = s_x + kBins + 1;                              // [n_mels]
    __shared__ double s_red[kNnlsThreads / 32];
    const int col = blockIdx.x;                               // (l, t)
    const int l = col / tb, t = col - l * tb;
    const int64_t row = static_cast<int64_t>(l) * T + t0 + t;
    for (int k = threadIdx.x; k < kBins; k += blockDim.x) {
        if (XMODE == 0) s_x[k] = static_cast<Real>(static_cast<const double*>(xv)[(static_cast<int64_t>(l) * kBins + k) * tb + t]);
        else { const Real sv = static_cast<Real>(static_cast<const float*>(xv)[row * ld_x + k]); s_x[k] = sv * sv; }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int m = warp; m < n_mels; m += nw) {                 // r[m] = sum_k A[m,k] x[k] - B[m]
        const float* a = basis + static_cast<int64_t>(m) * kBins;
        Real acc = 0;
        for (int k = lane; k < kBins; k += 32) acc = fma(static_cast<Real>(__ldg(a + k)), s_x[k], acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) {
            float b = mel[row * n_mels + m];
            if (is_log) b = expf(b);
            s_r[m] = acc - static_cast<Real>(b);
        }
    }
    __syncthreads();
    double pg = 0.0;
    for (int k = threadIdx.x; k < kBins; k += blockDim.x) {   // g[k] = inv_size * sum_m A[m,k] r[m]
        Real acc = 0;
        for (int m = 0; m < n_mels; ++m) acc = fma(static_cast<Real>(__ldg(basis + static_cast<int64_t>(m) * kBins + k)), s_r[m], acc);
        const double g = static_cast<double>(acc) * inv_size;
        if (grad) grad[(static_cast<int64_t>(l) * kBins + k) * tb + t] = g;
        // L-BFGS-B projgr with a lower bound only: g < 0 -> |g|, else min(x - 0, g)
        const double p = g < 0.0 ? -g : fmin(static_cast<double>(s_x[k]), g);
        pg = fmax(pg, p);
    }
    double v = 0.0;
    for (int m = threadIdx.x; m < n_mels; m += blockDim.x) v += static_cast<double>(s_r[m]) * static_cast<double>(s_r[m]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        pg = fmax(pg, __shfl_xor_sync(0xffffffffu, pg, o));
        v += __shfl_xor_sync(0xffffffffu, v, o);
    }
    // n_mels <= 256: the squares live in the first warps only; two small fixed-order reductions
    if (lane == 0) s_red[warp] = pg;
    __syncthreads();
    if (threadIdx.x == 0) {
        double mx = 0.0;
        for (int w = 0; w < nw; ++w) mx = fmax(mx, s_red[w]);
        pg_max[col] = mx;
    }
    __syncthreads();
    if (lane == 0) s_red[warp] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double sum = 0.0;
        for (int w = 0; w < nw; ++w) sum += s_red[w];
        value_parts[col] = 0.5 * inv_size * sum;
    }
}

// Screening pass (x_mode 2, no gradient wanted): the same projected-gradient sup-norm in float32, but BANDED -- the Slaney
// basis has ~2 non-zeros per bin (1,026 of 41,040 entries), and the dense kernel above re-reads all 164 KB of it from L2
// twice per column (2.1 GB for cfg3's 12,800 columns: 0.36 ms of a 3.7 ms Vocoder.infer call).  One WARP per column:
// lane <-> band for r = A x - B (the band's run of non-zeros), lane <-> bin for g = A^T r (the 1-3 bands covering the
// bin); ranges from a ctx table.  The caller repeats blocks within 10 % of the threshold in float64 with the dense kernel.
constexpr int kScreenWarps = 8;
constexpr int kScreenX = 520;   // per-warp x slot (513 used)

__global__ void __launch_bounds__(kScreenWarps * 32)
k_nnls_screen(const float* __restrict__ S, int64_t ld_x, const float* __restrict__ mel, int is_log,
              const float* __restrict__ basis, const int2* __restrict__ band_rng /*[n_mels] (first bin, count)*/,
              const int2* __restrict__ bin_rng /*[513] (first band, last band)*/, int n_mels, int n_pad, int64_t n_cols,
              int64_t T, int64_t t0, int tb, double inv_size, double* __restrict__ value_parts, double* __restrict__ pg_max) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t col = static_cast<int64_t>(blockIdx.x) * kScreenWarps + warp;
    if (col >= n_cols) return;                                   // (no CTA-wide barrier below)
    float* s_x = reinterpret_cast<float*>(smem_raw) + warp * (kScreenX + n_pad);
    float* s_r = s_x + kScreenX;
    const int64_t l = col / tb, t = col - l * tb;
    const int64_t row = l * T + t0 + t;
    for (int k = lane; k < kBins; k += 32) { const float sv = S[row * ld_x + k]; s_x[k] = sv * sv; }
    __syncwarp();
    double v = 0.0;
    for (int m = lane; m < n_mels; m += 32) {
        const int2 br = band_rng[m];
        const float* a = basis + static_cast<int64_t>(m) * kBins + br.x;
        const float* xs = s_x + br.x;
        float acc = 0.f;
        for (int i = 0; i < br.y; ++i) acc = fmaf(__ldg(a + i), xs[i], acc);
        float b = mel[row * n_mels + m];
        if (is_log) b = expf(b);
        const float r = acc - b;
        s_r[m] = r;
        v += static_cast<double>(r) * static_cast<double>(r);
    }
    __syncwarp();
    double pg = 0.0;
    for (int k = lane; k < kBins; k += 32) {
        const int2 mr = bin_rng[k];
        float acc = 0.f;
        for (int m = mr.x; m <= mr.y; ++m) acc = fmaf(__ldg(basis + static_cast<int64_t>(m) * kBins + k), s_r[m], acc);
        const double g = static_cast<double>(acc) * inv_size;
        const double p = g < 0.0 ? -g : fmin(static_cast<double>(s_x[k]), g);   // L-BFGS-B projgr, lower bound only
        pg = fmax(pg, p);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        pg = fmax(pg, __shfl_xor_sync(0xffffffffu, pg, o));
        v += __shfl_xor_sync(0xffffffffu, v, o);
    }
    if (lane == 0) { pg_max[col] = pg; value_parts[col] = 0.5 * inv_size * v; }
}

// The dense basis both kernels read and the banded view of it the screening kernel walks: per band its run of non-zero
// bins (first bin, count), then per bin the bands that cover it (first band, last band).
int nnls_init(spev_ctx* c) {
    const int n_mels = c->n_mels;
    const std::vector<float>& basis = c->h_basis;
    std::vector<int> rng(2 * static_cast<size_t>(n_mels) + 2 * kBins);
    for (int m = 0; m < n_mels; ++m) {
        int lo = kBins, hi = -1;
        for (int k = 0; k < kBins; ++k)
            if (basis[static_cast<size_t>(m) * kBins + k] != 0.f) { lo = std::min(lo, k); hi = std::max(hi, k); }
        rng[2 * m] = hi >= lo ? lo : 0;
        rng[2 * m + 1] = hi >= lo ? hi - lo + 1 : 0;
    }
    for (int k = 0; k < kBins; ++k) {
        int lo = n_mels, hi = -1;
        for (int m = 0; m < n_mels; ++m)
            if (basis[static_cast<size_t>(m) * kBins + k] != 0.f) { lo = std::min(lo, m); hi = std::max(hi, m); }
        rng[2 * n_mels + 2 * k] = hi >= lo ? lo : 0;
        rng[2 * n_mels + 2 * k + 1] = hi >= lo ? hi : -1;
    }
    int rc = upload(&c->d_basis, basis);
    return rc ? rc : upload(&c->d_nnls_rng, rng);
}

}  // namespace spev

using namespace spev;

extern "C" {

int spev_nnls_objective(spev_ctx* c, const void* x, int x_mode, int64_t ld_x, const float* mel, int is_log, int L, int64_t T,
                        int64_t t0, int tb, int size_cols, double* value_parts, double* grad, double* pg_max, void* stream) {
    SPEV_ON_CTX_DEVICE(c);
    SPEV_REQUIRE(x_mode >= 0 && x_mode <= 2, SPEV_E_INVALID, "spev_nnls_objective: x_mode must be 0, 1 or 2");
    SPEV_REQUIRE(x && mel && value_parts && pg_max, SPEV_E_INVALID, "nnls_objective: null argument");
    SPEV_REQUIRE(L > 0 && tb > 0 && t0 >= 0 && t0 + tb <= T, SPEV_E_INVALID, "nnls_objective: bad block [%lld, %lld) of %lld",
                 static_cast<long long>(t0), static_cast<long long>(t0 + tb), static_cast<long long>(T));
    const int x_is_f32_rows = x_mode != 0;            // 1: float64 arithmetic, 2: float32 screening pass
    SPEV_REQUIRE(!x_is_f32_rows || ld_x >= kBins, SPEV_E_INVALID, "nnls_objective: ld_x < 513");
    SPEV_REQUIRE(size_cols >= 0, SPEV_E_INVALID, "nnls_objective: size_cols < 0");
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    const double inv_size = 1.0 / (static_cast<double>(L) * c->n_mels * (size_cols > 0 ? size_cols : tb));      // 1 / B.size
    const size_t smem = sizeof(double) * (kBins + 1 + c->n_mels);
    const int grid = L * tb;
    if (x_mode == 2 && !grad && c->d_nnls_rng) {
        const int n_pad = (c->n_mels + 3) & ~3;
        const int64_t n_cols = static_cast<int64_t>(L) * tb;
        const size_t sm = sizeof(float) * kScreenWarps * (kScreenX + n_pad);
        const int2* rng = reinterpret_cast<const int2*>(c->d_nnls_rng);
        k_nnls_screen<<<static_cast<unsigned>((n_cols + kScreenWarps - 1) / kScreenWarps), kScreenWarps * 32, sm, st>>>(
            static_cast<const float*>(x), ld_x, mel, is_log, c->d_basis, rng, rng + c->n_mels, c->n_mels, n_pad, n_cols, T, t0, tb,
            inv_size, value_parts, pg_max);
    } else if (x_mode == 2)
        k_nnls_objective<1, float><<<grid, kNnlsThreads, smem, st>>>(x, ld_x, mel, is_log, c->d_basis, c->n_mels, L, T, t0, tb,
                                                                    inv_size, value_parts, grad, pg_max);
    else if (x_mode == 1)
        k_nnls_objective<1, double><<<grid, kNnlsThreads, smem, st>>>(x, ld_x, mel, is_log, c->d_basis, c->n_mels, L, T, t0, tb,
                                                                     inv_size, value_parts, grad, pg_max);
    else
        k_nnls_objective<0, double><<<grid, kNnlsThreads, smem, st>>>(x, 0, mel, is_log, c->d_basis, c->n_mels, L, T, t0, tb,
                                                                     inv_size, value_parts, grad, pg_max);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

}  // extern "C"
