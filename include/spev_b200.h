/* spev_b200.h -- C ABI of the B200-native spectral hot path for SPEV-TTS.
 *
 * The reference (DhrG23/spev-tts) has no FFI/plugin interface: its boundary for this path is
 * a handful of Python call sites (file:line are in /root/reference/).  Each entry point below
 * names the reference call it replaces; the Python shims in spev_tts_b200/ keep the
 * reference's own signatures on top of this ABI (INTEGRATION.md shows the ctypes binding).
 *
 * Conventions
 *   - every pointer marked "dev" is device memory on the ctx's GPU; "host" is host memory.
 *   - the caller owns every buffer (inputs, outputs, workspace).  The library allocates only
 *     ctx-owned constants in spev_create and frees them in spev_destroy.
 *   - all work is enqueued asynchronously on `stream` (a cudaStream_t passed as void*); no
 *     entry point synchronises.
 *   - return value 0 = ok, negative = error (SPEV_E_*); text via spev_last_error()
 *     (thread-local).  No C++ exception crosses the ABI.  There is NO CPU fallback: without
 *     an sm_100 device spev_create fails with SPEV_E_DEVICE.
 *   - batches are "flat": items (utterances / spectrograms) are concatenated and described by a
 *     frame prefix-offset array plus per-CTA tile tables built on the host by spev_plan_*_tiles().
 */
#ifndef SPEV_B200_H
#define SPEV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPEV_ABI_VERSION 1

#if defined(__GNUC__)
#define SPEV_API __attribute__((visibility("default")))
#else
#define SPEV_API
#endif

#define SPEV_OK 0
#define SPEV_E_INVALID (-1)     /* bad argument */
#define SPEV_E_UNSUPPORTED (-2) /* configuration outside what the kernels implement */
#define SPEV_E_DEVICE (-3)      /* no sm_100 device / wrong device */
#define SPEV_E_CUDA (-4)        /* CUDA runtime error (message has the cudaError string) */
#define SPEV_E_WORKSPACE (-5)   /* workspace too small */

#define SPEV_TILE_FRAMES 32 /* frames per CTA tile (STFT-type kernels); == spev_tile_frames() */
#define SPEV_TILE_CHUNKS 29 /* 256-sample output chunks per CTA tile (ISTFT); == spev_tile_chunks() */
#define SPEV_SPEC_LD 520    /* row pitch (elements) of internal [F,513] spectra */

typedef struct spev_ctx spev_ctx;

/* One CTA tile.  Built on the host (spev_plan_frame_tiles / spev_plan_chunk_tiles) so that a
 * kernel needs exactly one 48-byte read per tile and no dependent look-ups.
 *  frame tile (STFT-type kernels): `n` (<= SPEV_TILE_FRAMES) consecutive frames t0.. of one item.
 *     src0 = absolute index, in the flat sample buffer, of the first staged sample
 *            (= lo + hop*t0 - n_fft/2; may lie before lo: centre padding reads as zero)
 *     lo, hi = absolute bounds of the item's samples (zero outside)
 *     row0 = global index (row of the [F, .] outputs) of frame t0
 *  chunk tile (ISTFT): `n` (<= SPEV_TILE_CHUNKS) consecutive hop-sized output chunks t0.. .
 *     src0 = absolute index in y of the first output sample of chunk t0
 *     row0 = global row of item frame (t0 - 1): the first of the n+3 frames the tile gathers
 *            (one before the item's first row when t0 == 0; never dereferenced then)
 *     lo, hi unused. */
typedef struct spev_tile {
    int64_t src0, lo, hi, row0;
    int32_t n, t0, T /* frames in the item */, item;
} spev_tile;

/* Flat batch descriptor.  Item i owns rows [frame_off[i], frame_off[i+1]) of every [F, .] array.
 * Framing is librosa center=True: an item of N samples has T = 1 + N / hop frames; an ISTFT
 * output item has (T-1)*hop samples at offset hop*(frame_off[i] - i). */
typedef struct spev_batch {
    int32_t n_items;
    int32_t n_ftiles;
    int32_t n_ctiles;          /* may be 0 when no ISTFT is requested */
    int32_t reserved;
    int64_t n_frames;          /* == frame_off[n_items] */
    const int64_t* frame_off;  /* dev [n_items+1] */
    const spev_tile* ftiles;   /* dev [n_ftiles] */
    const spev_tile* ctiles;   /* dev [n_ctiles] */
} spev_batch;

SPEV_API int spev_abi_version(void);
SPEV_API const char* spev_last_error(void);
SPEV_API int spev_tile_frames(void); /* tile sizes the loaded library was built with */
SPEV_API int spev_tile_chunks(void);

/* ctx: immutable after creation, one per device, shareable between host threads.
 * Owns the periodic Hann window, FFT twiddles, the Slaney mel basis keyed on
 * (sr, n_fft, n_mels, fmin, fmax) in dense + banded form, and its pseudo-inverse.
 * fmax <= 0 means sr/2 (librosa's fmax=None).  This round supports n_fft = win = 1024,
 * hop = 256 (the reference CONFIG, spev_real_metrics.py:60-67); anything else returns
 * SPEV_E_UNSUPPORTED.   Replaces: librosa.filters.mel / get_window under :363 and :730-733. */
SPEV_API int spev_create(spev_ctx** out, int device, int sr, int n_fft, int hop, int win, int n_mels,
                float fmin, float fmax);
SPEV_API void spev_destroy(spev_ctx* ctx);

/* Host copies of ctx constants (tests, INTEGRATION).  basis: [n_mels*513], pinv: [513*n_mels]
 * (row-major), window: [n_fft]. */
SPEV_API int spev_get_mel_basis(const spev_ctx* ctx, float* basis_host);
SPEV_API int spev_get_mel_pinv(const spev_ctx* ctx, float* pinv_host);
SPEV_API int spev_get_window(const spev_ctx* ctx, float* window_host);

/* Host-only (no GPU needed): the float32 Slaney basis [n_mels, 1+n_fft/2] exactly as the ctx
 * builds it, and the float64-Jacobi pseudo-inverse [n, m] of a row-major [m, n] matrix. */
SPEV_API int spev_host_mel_basis(int sr, int n_fft, int n_mels, float fmin, float fmax, float* basis);
SPEV_API int spev_host_pinv(const float* a, int m, int n, float* pinv);

/* Host helpers that build the tile tables (call with out == NULL to get the count).
 *   frames[i]     : frames of item i
 *   sample_lo[i]  : absolute start of item i's samples in the flat buffer, n_samples[i] its
 *                   length (waveform batches: spev_logmel / spev_stft_power); pass NULL for both
 *                   to describe the implicit ISTFT-output layout (spev_stft, spev_gl_*, where
 *                   item i has (T_i-1)*hop samples at hop*(frame_off[i]-i)). */
SPEV_API int64_t spev_plan_frame_tiles(const int64_t* frames, const int64_t* sample_lo,
                                       const int64_t* n_samples, int n_items, spev_tile* out);
SPEV_API int64_t spev_plan_chunk_tiles(const int64_t* frames, int n_items, spev_tile* out);

/* STFT -> |.|^2 -> mel -> (optional) log compression, fused, one launch.
 *   samples : dev float32, flat buffer the frame tiles index into
 *   out     : dev float32 [n_frames, n_mels] row-major  (== the reference's cache layout
 *             `mel.T`, spev_real_metrics.py:421)
 *   mode 0  : mel power            (librosa.feature.melspectrogram, :363)
 *   mode 1  : clamp(log(max(mel, floor)), lo, hi)   (:364-366; reference: 1e-5, -10, 2)
 * Replaces spev_real_metrics.py:363-367. */
SPEV_API int spev_logmel(spev_ctx* ctx, const spev_batch* batch, const float* samples, float* out,
                int mode, float floor, float lo, float hi, void* stream);

/* 16-bit PCM -> float32, out[i] = pcm[i] / 32768 (exact): the values soundfile / librosa.load hand to
 * melspectrogram for a 16-bit wav (spev_real_metrics.py:332 -> :363).  Lets a cache build ship PCM
 * over PCIe (half the bytes) and widen on the device. */
SPEV_API int spev_pcm16_to_f32(const int16_t* pcm, int64_t n, float* out, void* stream);

/* Same front end, but writes the power spectrum |STFT|^2 as [n_frames, SPEV_SPEC_LD] (pad
 * columns zero) -- the A operand of spev_mel_project. */
SPEV_API int spev_stft_power(spev_ctx* ctx, const spev_batch* batch, const float* samples, float* power,
                    void* stream);

/* Tensor-core (tcgen05, 3xTF32, TMA-staged) mel projection  power[F,513] . basis^T -> [F,n_mels]
 * with the same epilogue modes as spev_logmel.  Replaces the einsum inside
 * librosa.feature.melspectrogram (:363) + :364-366. */
SPEV_API int spev_mel_project(spev_ctx* ctx, const float* power, int64_t n_frames, float* out, int mode,
                     float floor, float lo, float hi, void* stream);

/* mel -> linear magnitude: S = sqrt(max(pinv(basis) . M, 0)), the warm start that librosa's
 * NNLS (util.nnls, L-BFGS-B) returns unchanged for reference-range inputs (SURVEY 0.5).
 *   mel     : dev float32.  layout 0: [n_frames, n_mels] frame-major flat;
 *             layout 1: per item [n_mels, T_i] at element offset frame_off[i]*n_mels
 *             (the reference's Vocoder.infer input, :725-733)
 *             layout 0 runs on the tensor cores (TMA + tcgen05 3xTF32, TMEM accumulators);
 *             layout 1 on an FFMA kernel
 *   is_log  : 1 -> apply exp() first (:729)
 *   S       : dev float32 [n_frames, ld_s]
 * Replaces librosa.feature.inverse.mel_to_stft under :730. */
SPEV_API int spev_mel_to_mag(spev_ctx* ctx, const spev_batch* batch, const float* mel, int layout,
                    int is_log, float* S, int64_t ld_s, void* stream);

/* A/B switch for the tensor-core path of spev_mel_to_mag (default on): 0 forces the FFMA kernel. */
SPEV_API int spev_set_tensor_core(spev_ctx* ctx, int enable);

/* Objective of librosa.util.nnls (the solver inside librosa.feature.inverse.mel_to_stft, spev_real_metrics.py:730) for
 * one block of tb columns starting at column t0 of L stacked items of T columns each:
 *     f(x) = 0.5 / size * || A x - B ||^2,   grad = A^T (A x - B) / size,   size = L * n_mels * (size_cols ? size_cols : tb)
 *     (size_cols lets one launch cover several of librosa's equal-sized blocks: tb = their total, size_cols = one block),
 * evaluated in float64 like librosa's (scipy hands its objective a float64 x); A = the ctx's mel basis, B = mel columns.
 *   x        : x_mode 0: device float64 [L, 513, tb] (librosa's own element order);
 *              x_mode 1: device float32 magnitude rows S [L*T, ld_x] as written by spev_mel_to_mag -> x = S^2 (the warm start);
 *              x_mode 2: as 1, but the arithmetic in float32 -- a cheap screening pass; re-evaluate blocks whose pg_max lies
 *                        within 10 % of pgtol with x_mode 1 before deciding
 *   mel      : device float32 [L*T, n_mels] frame-major mel power (or log-mel with is_log != 0)
 *   value_parts [L*tb] float64: per-column share of f (f = their sum, column order (l, t));
 *   grad     [L, 513, tb] float64 or NULL;   pg_max [L*tb]: per-column max |projected gradient| for the bound x >= 0
 *              (L-BFGS-B's convergence measure: it returns the start point when max(pg_max) <= pgtol = 1e-5). */
SPEV_API int spev_nnls_objective(spev_ctx* ctx, const void* x, int x_mode, int64_t ld_x, const float* mel, int is_log,
                                 int L, int64_t T, int64_t t0, int tb, int size_cols, double* value_parts, double* grad,
                                 double* pg_max,
                                 void* stream);

/* ISTFT (irFFT-1024, Hann, gather overlap-add, window-sum-square normalisation).
 *   spec : dev float2 [n_frames, ld] ; y : dev float32, item i at 256*(frame_off[i]-i),
 *   length (T_i-1)*256.   Replaces librosa.istft inside griffinlim (:730-733). */
SPEV_API int spev_istft(spev_ctx* ctx, const spev_batch* batch, const void* spec, int64_t ld, float* y,
               void* stream);

/* STFT of y (same item layout as spev_istft's output) -> spec [n_frames, ld] float2. */
SPEV_API int spev_stft(spev_ctx* ctx, const spev_batch* batch, const float* y, void* spec, int64_t ld,
              void* stream);

/* One Griffin-Lim phase update (the body of librosa.griffinlim's loop after the istft):
 *   reb = STFT(y); a = reb - alpha*tprev (skipped when has_prev == 0);
 *   ang = S * a / (|a| + tiny);  tprev <- reb (in place).
 * ang, tprev: dev float2 [n_frames, ld]; S: dev float32 [n_frames, ld_s]. */
SPEV_API int spev_gl_phase_update(spev_ctx* ctx, const spev_batch* batch, const float* y, const float* S,
                         int64_t ld_s, void* ang, void* tprev, int64_t ld, float alpha,
                         int has_prev, void* stream);

/* Full Griffin-Lim: ang0 = S*exp(i*phase); n_iter x (istft, stft + phase update); final istft -- executed as
 * istft once, then n_iter x (fused stft + phase update + inverse transform of the new spectra, pair overlap-add).
 * Same arithmetic per frame as spev_istft / spev_gl_phase_update, except that the phase normalisation uses a 2-ulp
 * rsqrt and the <= 4 overlap-add terms of a sample are summed pair by pair: agrees with those entry points to rounding.
 *   init_phase : dev float32 [n_frames, 513] radians, or NULL -> 2*pi*U[0,1) from `seed`
 *   y          : dev float32 [256*(n_frames - n_items)]
 *   workspace  : dev, >= spev_griffinlim_workspace_bytes(n_frames)
 * Replaces librosa.griffinlim under spev_real_metrics.py:730-733 (n_iter default 32 there,
 * momentum 0.99). */
SPEV_API size_t spev_griffinlim_workspace_bytes(int64_t n_frames);
SPEV_API int spev_griffinlim(spev_ctx* ctx, const spev_batch* batch, const float* S, int64_t ld_s,
                    const float* init_phase, uint64_t seed, int n_iter, float momentum, float* y,
                    void* workspace, size_t workspace_bytes, void* stream);

/* Frame-level energy / brightness (SURVEY 8(f) row 1).  For every frame t (hop 256) of the centre-padded
 * 2048-sample window:  rms[t] = sqrt(mean(x^2))  and  centroid[t] = sum_k f_k|X_k| / sum_k|X_k|,
 * X = rFFT-2048(hann * x), f_k = k*sr/2048.  Same flat waveform batch as spev_logmel; outputs [n_frames].
 * Replaces librosa.feature.rms(y, hop_length=256) and librosa.feature.spectral_centroid(y, sr,
 * hop_length=256) at spev_real_metrics.py:370-371 (the caller takes the logs). */
SPEV_API int spev_frame_features(spev_ctx* ctx, const spev_batch* batch, const float* samples, float* rms,
                                 float* centroid, void* stream);

/* Per-phoneme pooling of a frame-level curve: for phoneme p of item i with duration d_p frames,
 *   out[p] = clamp((mean(curve[frame_off[i] + start_p .. + d_p)) - mu) / sigma, lo, hi)
 * where start_p is the running sum of the item's earlier durations.  durs: dev int64 flat, item i
 * owns [phone_off[i], phone_off[i+1]).  Replaces the e / bri (and, with mu=1, sigma=-1, br) lines of
 * the per-phone loop, spev_real_metrics.py:400-417. */
SPEV_API int spev_segment_pool(const float* curve, const int64_t* frame_off, const int64_t* durs,
                               const int64_t* phone_off, int n_items, float mu, float sigma, float lo, float hi,
                               float* out, void* stream);
/* Same, pooling log(curve + log_eps): the reference takes np.log(rms + 1e-6) / np.log(cent + 1e-8) per frame
 * (spev_real_metrics.py:370, :397) before the per-phone mean. */
SPEV_API int spev_segment_pool_log(const float* curve, float log_eps, const int64_t* frame_off, const int64_t* durs,
                                   const int64_t* phone_off, int n_items, float mu, float sigma, float lo, float hi,
                                   float* out, void* stream);

/* GPU-side batching of a resident cache (SURVEY 8(f) row 3): ragged -> zero-padded copies, i.e. the
 * pad_sequence(..., batch_first=True) calls of the reference's collate_fn (spev_real_metrics.py:449-462)
 * for up to 12 arrays in one launch.  Array k holds rows of row_bytes bytes, indexed per frame
 * (per_phone = 0: item i owns rows [frame_off[i], frame_off[i+1])) or per phoneme (per_phone = 1:
 * phone_off).  For batch entry b (item sel[b], or b when sel is NULL):
 *   dst_k[b, r, :] = src_k[off[item] + r, :]  for r < len(item),  0 for len(item) <= r < t_max / p_max.
 * Rows are copied verbatim: bit-exact for every dtype. */
typedef struct spev_pad_array {
    const void* src;     /* dev: flat [rows, row_bytes] */
    void* dst;           /* dev: [B, t_max or p_max, row_bytes] */
    int64_t row_bytes;
    int32_t per_phone;
    int32_t reserved;
} spev_pad_array;
SPEV_API int spev_collate(const spev_pad_array* arrays_host, int n_arrays, const int64_t* frame_off,
                          const int64_t* phone_off, const int64_t* sel, int B, int64_t t_max, int64_t p_max,
                          void* stream);

/* Batched 2-D transpose, dst[b][c][r] = src[b][r][c] (pitches and batch strides in ELEMENTS of elem_bytes = 4 or 8):
 * the layout change between librosa's [..., bins, T] arrays (the shapes at spev_real_metrics.py:363 and :730-733) and
 * the frame-major rows [F, pitch] the kernels work on, e.g. a [b, 80, T] mel -> rows [b*T, 80], or magnitude rows
 * [b*T, 520] -> [b, 513, T] (rows = T, cols = 513, src_pitch = 520). */
SPEV_API int spev_transpose_batched(const void* src, void* dst, int elem_bytes, int64_t batches, int rows, int cols,
                                    int64_t src_pitch, int64_t src_batch, int64_t dst_pitch, int64_t dst_batch,
                                    void* stream);

/* Segmented device copy: dst[dst_off[i] .. +nbytes[i]) = src[src_off[i] .. +nbytes[i]) for n_segments runs of bytes
 * (all tables on the device; piece_off[i] = first 16 KB piece of segment i, piece_off is the exclusive prefix sum of
 * ceil(nbytes[i] / spev_copy_segments_piece_bytes()), n_pieces its total).  Used to put gathered cache shards
 * (rank-major rows) into corpus order and to pack utterances into shards: the GPU form of the per-utterance
 * `'mel': mel.T.clone()` stores of spev_real_metrics.py:419-425. */
SPEV_API int spev_copy_segments_piece_bytes(void);
SPEV_API int spev_copy_segments(const void* src, void* dst, const int64_t* src_off, const int64_t* dst_off,
                                const int64_t* nbytes, const int64_t* piece_off, int n_segments, int64_t n_pieces,
                                void* stream);

/* Cap the number of CTAs the persistent FFT kernels launch (default: one per SM).  A multi-GPU cache build that
 * overlaps the NCCL gather of finished chunks with the kernel of the next chunk leaves a few SMs to NCCL's
 * send/recv kernels this way (the FFT CTAs each fill a whole SM).  max_ctas = 0 restores the default. */
SPEV_API int spev_set_sm_limit(spev_ctx* ctx, int max_ctas);

/* LengthRegulator, phase 1: sanitise durations (non-finite / <0 / >1000 -> 0, truncate),
 * inclusive row cumsum, mel_lens = max(total, 1), max_len = max(mel_lens).
 *   dur       : dev [B,T], dur_dtype 0=int64 1=int32 2=float32 3=float64 4=float16 5=bfloat16
 *   cumsum    : dev int32 [B,T]
 *   mel_lens  : dev int64 [B]
 *   max_len_dev  : dev int64 [1];  max_len_host : pinned host int64 [1] or NULL (async copy;
 *                  the caller synchronises the stream once before reading it)
 * Replaces the validation loop of LengthRegulator.forward, spev_real_metrics.py:126-142. */
SPEV_API int spev_lr_plan(const void* dur, int dur_dtype, int B, int T, int32_t* cumsum, int64_t* mel_lens,
                 int64_t* max_len_dev, int64_t* max_len_host, void* stream);

/* LengthRegulator, phase 2: out[b,f,:] = x[b, idx(b,f), :] for f < total_b else 0, where
 * idx = searchsorted(cumsum[b], f, right).  Rows are copied verbatim (row_bytes = H*itemsize),
 * so any dtype is bit-exact.  Replaces repeat/cat/pad/stack, :135-146 (and expand_feat,
 * :228-236, with row_bytes = itemsize). */
SPEV_API int spev_lr_expand(const void* x, int64_t row_bytes, const int32_t* cumsum, int B, int T,
                   void* out, int64_t max_len, void* stream);

/* Fused expand of the hidden states plus n_feat scalar curves in one launch (the six
 * LengthRegulator calls of RealMetricsFastSpeech2.forward, :226-236, with the post-clamps of
 * :239-243 applied when clamp_lo/hi are non-NULL).
 *   feats : dev float32 [n_feat, B, T];  feats_out : dev float32 [n_feat, B, max_len] */
SPEV_API int spev_lr_expand_fused(const void* x, int64_t row_bytes, const float* feats, int n_feat,
                         const float* clamp_lo_host, const float* clamp_hi_host,
                         const int32_t* cumsum, int B, int T, void* out, float* feats_out,
                         int64_t max_len, void* stream);

/* Fused variance adaptor (SURVEY 8(f) row 4): the whole block spev_real_metrics.py:226-252 in one launch --
 * expand x by the durations, expand + clamp the n_feat scalar curves, apply each curve's
 * Conv1d(1 -> H, kernel 3, padding 1) embedding and add the embeddings to the expanded hidden states:
 *   out[b,f,:] = x[b,idx(b,f),:] + sum_j ( bias_j + w_j[:,0]*cv_j[b,f-1] + w_j[:,1]*cv_j[b,f] + w_j[:,2]*cv_j[b,f+1] )
 *   x [B,T,H] float32; feats [n_feat,B,T]; conv_w [n_feat,H,3] (= nn.Conv1d.weight[:,0,:] per curve);
 *   conv_b [n_feat,H]; cumsum from spev_lr_plan; out [B,max_len,H]; feats_out [n_feat,B,max_len] or NULL. */
SPEV_API int spev_variance_fuse(const float* x, const float* feats, int n_feat, const float* clamp_lo_host,
                                const float* clamp_hi_host, const float* conv_w, const float* conv_b,
                                const int32_t* cumsum, int B, int T, int H, float* out, float* feats_out,
                                int64_t max_len, void* stream);

/* Backward of spev_lr_expand / spev_lr_expand_fused: the autograd of the reference's repeat / cat / pad / stack
 * (spev_real_metrics.py:135-146), which its Trainer differentiates through (loss.backward(), :574).
 *   grad_x[b,t,:]     = sum over the frames f of segment t (cumsum[t-1] <= f < cumsum[t]) of grad_out[b,f,:]
 *   grad_feats[j,b,t] = pass_j(feats[j,b,t]) * sum over segment t of grad_feats_out[j,b,f]
 * pass_j = (lo_j <= v <= hi_j), torch.clamp's backward mask, when clamp_lo/hi are given (then `feats`, the
 * forward's curves, is required); padding frames belong to no segment.  Every output element has one owner
 * thread that adds its frames in ascending order: no atomics, bit-reproducible.
 *   grad_out [B,max_len,H] / grad_x [B,T,H] of dtype 0=float32 1=float64 2=float16 3=bfloat16 (NULL,NULL: skip)
 *   grad_feats_out [n_feat,B,max_len] / grad_feats [n_feat,B,T] float32 (n_feat = 0: skip) */
SPEV_API int spev_lr_expand_backward(const void* grad_out, int dtype, int H, const float* grad_feats_out, int n_feat,
                                     const float* feats, const float* clamp_lo_host, const float* clamp_hi_host,
                                     const int32_t* cumsum, int B, int T, int64_t max_len, void* grad_x,
                                     float* grad_feats, void* stream);

/* Backward of spev_variance_fuse (the autograd of spev_real_metrics.py:226-252: six LengthRegulator calls, five
 * clamps, five Conv1d(1,H,3,padding=1) embeddings, their sum).  Any of the four outputs may be NULL.
 *   grad_out [B,max_len,H];  grad_x [B,T,H];  grad_feats [n_feat,B,T];  grad_w [n_feat,H,3];  grad_b [n_feat,H]
 * n_feat <= 5, H <= 1024.  Deterministic (per-CTA partial sums added in CTA order).  Workspace: caller-owned device
 * memory of spev_variance_fuse_backward_workspace_bytes(). */
SPEV_API size_t spev_variance_fuse_backward_workspace_bytes(int n_feat, int B, int H, int64_t max_len);
SPEV_API int spev_variance_fuse_backward(const float* grad_out, const float* feats, int n_feat, const float* clamp_lo_host,
                                         const float* clamp_hi_host, const float* conv_w, const int32_t* cumsum, int B,
                                         int T, int H, int64_t max_len, float* grad_x, float* grad_feats, float* grad_w,
                                         float* grad_b, void* workspace, size_t workspace_bytes, void* stream);

/* Inference duration rule, spev_real_metrics.py:215:
 *   dur = (int64) rint(clamp((exp(log_dur) - 1) * d_control, 0, 500))   (round-half-even) */
SPEV_API int spev_duration_rule(const float* log_dur, int64_t n, float d_control, int64_t* dur,
                       void* stream);

/* Bucketize + embedding lookup (canonical FastSpeech 2 variance embedding; no reference site,
 * semantics = torch.bucketize(right) + F.embedding, SURVEY a-13).
 *   idx_out : dev int64 [n] or NULL;  out : dev float32 [n,H] or NULL;
 *   accumulate != 0 -> out += table[idx] */
SPEV_API int spev_bucketize_embed(const float* v, int64_t n, const float* boundaries, int n_boundaries,
                         int right, const float* table, int H, int64_t* idx_out, float* out,
                         int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------------
 * pYIN  (SURVEY 8(f) "next" row 2)
 * Replaces  f0, _, voiced_prob = librosa.pyin(y, fmin=60, fmax=500, sr=22050, hop_length=256)
 * at /root/reference/spev_real_metrics.py:369 (cache build) and :311 (statistics pass): librosa defaults
 * frame_length=2048, win_length=1024, 100 thresholds, beta(2,18), Boltzmann(2), 10-cent bins,
 * max_transition_rate=35.92 octaves/s, switch_prob=0.01, no_trough_prob=0.01, centre zero padding.
 * Three stages so that each can be checked on its own; frames are addressed through the same
 * spev_batch frame tiles as spev_logmel (item i has 1 + len_i/256 frames).
 * ---------------------------------------------------------------------------------------------- */
typedef struct spev_pyin spev_pyin;
/* hop_length: 256 (cache loop, :369) or 512 (librosa's default frame_length/4, used by the statistics pass
 * :311).  It sets the transition band (max_transition_rate * hop / sr); stages 1-2 run on the hop-256 frame
 * grid and the caller keeps every (hop_length/256)-th frame before stage 3.
 * beta_probs_host: optional host array [100] = diff(beta(2,18).cdf(linspace(0,1,101))) as the caller's own
 * statistics library rounds it (the Python shim passes scipy's, i.e. librosa's exact table); NULL = built-in
 * closed form (equal to ~1e-16 absolute). */
SPEV_API int spev_pyin_create(spev_pyin** out, int device, int sr, int hop_length, float fmin, float fmax,
                              const double* beta_probs_host);
SPEV_API void spev_pyin_destroy(spev_pyin* ctx);
/* n_bins: voiced pitch bins (states = 2*n_bins); lags min_period..max_period (n_lags of them). */
SPEV_API int spev_pyin_info(const spev_pyin* ctx, int* n_bins, int* min_period, int* max_period, int* n_lags);
/* Host copies of the model tables: dense log(transition + tiny) [2*n_bins, 2*n_bins] (row = from-state),
 * bin frequencies [n_bins], beta-distributed threshold weights [100].  Any pointer may be NULL. */
SPEV_API int spev_pyin_host_tables(const spev_pyin* ctx, double* log_transition, double* freqs, double* beta_probs);
/* Stage 1: cumulative-mean-normalised difference.  samples: device f32 (flat batch), yin: device f32
 * [n_frames, n_lags]  (librosa.core.pitch._cumulative_mean_normalized_difference). */
SPEV_API int spev_pyin_cmnd(spev_pyin* ctx, const spev_batch* batch, const float* samples, float* yin, void* stream);
/* Stage 2: trough statistics -> log observation probabilities (librosa.core.pitch.__pyin_helper).
 * logobs f32 [n_frames, n_bins] = log(P(voiced bin) + tiny); log_unvoiced f32 [n_frames] = the (uniform)
 * log-probability of each unvoiced state; voiced_prob f32 [n_frames]. */
SPEV_API int spev_pyin_observe(spev_pyin* ctx, const float* yin, int64_t n_frames, float* logobs,
                               float* log_unvoiced, float* voiced_prob, void* stream);
/* Stage 3: Viterbi decode per item (librosa.sequence.viterbi) + state -> (f0, voiced_flag).
 * frame_off: device int64 [n_items+1]; states int32 [n_frames]; f0 f32 [n_frames] (NaN where unvoiced)
 * and voiced_flag u8 [n_frames] may be NULL.  workspace: device, >= spev_pyin_decode_workspace_bytes. */
SPEV_API size_t spev_pyin_decode_workspace_bytes(const spev_pyin* ctx, int64_t n_frames);
SPEV_API int spev_pyin_decode(spev_pyin* ctx, const float* logobs, const float* log_unvoiced, const int64_t* frame_off,
                              int n_items, int64_t n_frames, int32_t* states, float* f0, uint8_t* voiced_flag,
                              void* workspace, size_t workspace_bytes, void* stream);

/* Per-phoneme pitch statistics from the decoded states, spev_real_metrics.py:399-414 (float64 like numpy):
 *   f0_log = log(f0 + 1e-8) on voiced frames (state < n_bins); unvoiced frames are masked (the reference's
 *   log(1e-8 + 1e-8) < -5 test);  pitch[p] = clip((mean - p_mean) / p_std, lo, hi), or clip(0) without voiced
 *   frames;  rough[p] = clip(population std, 0, rough_hi), 0 without voiced frames.
 *   states int32 [F]; frame_off / phone_off int64 [n_items+1]; durs int64 [P]; pitch, rough f32 [P]. */
SPEV_API int spev_pitch_pool(const spev_pyin* ctx, const int32_t* states, const int64_t* frame_off, const int64_t* durs,
                             const int64_t* phone_off, int n_items, double p_mean, double p_std, float lo, float hi,
                             float rough_hi, float* pitch, float* rough, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SPEV_B200_H */
