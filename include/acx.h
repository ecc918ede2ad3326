/*
 * libacx -- C ABI of the B200-native audioset-convnext inference hot path.
 *
 * The reference (topel/audioset-convnext-inf) is pure Python/PyTorch and has NO FFI, plugin
 * or operator interface: its boundary is the Python class API of
 *   src/audioset_convnext_inf/pytorch/convnext.py  (ConvNeXt.forward :287-331,
 *   forward_scene_embeddings :333-366, forward_frame_embeddings :369-402).
 * This header is therefore the interface a maintainer of the reference would bind with
 * ctypes underneath those three methods (see INTEGRATION.md); every entry point cites the
 * reference lines whose computation it replaces.
 *
 * Conventions
 *  - plain pointers and sizes only; all pointers are DEVICE pointers unless suffixed _host.
 *  - every call is asynchronous on `stream` (a cudaStream_t passed as void*), never
 *    synchronises, never allocates persistent device memory; the caller (torch) owns all
 *    buffers, including the workspace.
 *  - return 0 on success, non-zero ACX_ERR_* otherwise; acx_last_error() gives the message
 *    (thread-local).  No C++ exceptions cross this boundary.
 *  - activations are channels-last (N, H, W, C) with H = time, W = mel;
 *    `act_dtype` = ACX_BF16 (tensor-core path) or ACX_F32 (fp32-accurate SIMT path).
 */
#ifndef ACX_H_
#define ACX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACX_VERSION 100
#define ACX_API __attribute__((visibility("default")))

enum { ACX_OK = 0, ACX_ERR_ARG = 1, ACX_ERR_CUDA = 2, ACX_ERR_UNSUPPORTED = 3, ACX_ERR_WORKSPACE = 4 };
enum { ACX_BF16 = 0, ACX_F32 = 1 };

/* GEMM epilogues (acx_gemm). */
enum {
  ACX_EPI_BIAS = 0,            /* out = acc + bias[n]                                  (CX:231-234 conv) */
  ACX_EPI_BIAS_GELU = 1,       /* out = gelu_erf(acc + bias[n])                         (CX:79-80)        */
  ACX_EPI_BIAS_SCALE_RESID = 2 /* out = resid[m,n] + gamma[n] * (acc + bias[n])         (CX:81-86)        */
};

ACX_API int acx_version(void);
ACX_API const char* acx_last_error(void);
/* 1 if the current device is compute capability 10.x (B200), else 0 (and sets last error). */
ACX_API int acx_device_ok(void);

/* ---- front end: torchlibrosa Spectrogram + LogmelFilterBank + bn0 (CX:298-306) ------------- */

/* Split-precision operands of the tensor-core DFT are FP16 pairs of the value scaled by 2^ACX_FE_SCALE_LOG2
 * (hi = fp16(s x), lo = fp16(s x - hi): 22 mantissa bits, lo stays a normal fp16 down to |x| ~ 5e-4). */
#define ACX_FE_SCALE_LOG2 8

/* Reflect-pad n_fft/2 both sides (torchlibrosa STFT.forward: F.pad(..., mode='reflect')) and
 * split each fp32 sample into the scaled fp16 hi + lo pair above.  wave (B, L) fp32 ->
 * hi, lo (B, ld_pad) fp16 with ld_pad >= L + n_fft, ld_pad % 8 == 0.  If act_dtype == ACX_F32
 * writes one fp32 padded (unscaled) array to `hi` and ignores `lo`. */
ACX_API int acx_wave_prep(const float* wave, void* hi, void* lo, int B, int L, int n_fft, int ld_pad,
                  int act_dtype, void* stream);

/* Same, reading int16 PCM (the AudioSet HDF5 storage format, reference utils/data_generator.py:70-74) and
 * converting x / 32767. on the fly (utils/utilities.py:226-227): halves the H2D bytes of the eval loop. */
ACX_API int acx_wave_prep_pcm16(const int16_t* pcm, void* hi, void* lo, int B, int L, int n_fft, int ld_pad,
                        int act_dtype, void* stream);

/* fp32-accurate path: spec (B*T, 2*n_bins) fp32 (re | im, from acx_gemm_f32 on the padded wave)
 * -> power -> mel (sparse band form) -> 10*log10(max(.,1e-10)) -> bn0 affine.
 * mel_lo/mel_hi (n_mels) int32 give each filter's non-zero bin range [lo, hi); melT is
 * (n_mels, n_bins) fp32 (transposed melW); bn_scale/bn_shift (n_mels) fold bn0 (eps 1e-5). */
ACX_API int acx_power_mel_log(const float* spec, int ld_spec, int n_bins, const float* melT, const int32_t* mel_lo,
                      const int32_t* mel_hi, const float* bn_scale, const float* bn_shift, float* out,
                      int rows, int n_mels, void* stream);

/* tensor-core path: one fused kernel, frames x DFT (split-fp16 x3, fp32 accumulate in TMEM) ->
 * power -> x mel (split-bf16 x3) -> log10 -> bn0; never writes the spectrogram to HBM.
 * hi/lo: padded split waveform from acx_wave_prep.  dft_hi/lo: (n_chunks*128, n_fft) fp16 pairs of the
 * 2^ACX_FE_SCALE_LOG2-scaled windowed-DFT rows,
 * chunk c rows [0,64) = real rows of bins [64c, 64c+64), rows [64,128) = imag rows.
 * mel_hi/lo: (n_chunks*256, 64) bf16, chunk c rows m<224 = melW[64c + k, m] (K-major), rest 0.
 * out (B, T, n_mels) fp32. */
/* The same front end on FOLDED frames (frontend_folded.cu): for STFT rows with the real-input symmetry of a periodic-Hann
 * windowed DFT (W_re even, W_im odd about n = n_fft/2, zero at n = 0; torchlibrosa Spectrogram, CX:179-187) a frame's
 * spectrum is  re = E . Wre'^T, im = O . Wim'^T  with E[0] = x[512], E[j] = x[j] + x[1024-j], O[0] = 0, O[j] = x[j] - x[1024-j]:
 * half the tensor-core work of the dense product.
 *   acx_frame_fold(_pcm16): waveform (B, L) fp32 / int16 PCM -> f_hi / f_lo (B, T, n_fft) fp16 pairs of the
 *     2^ACX_FE_SCALE_LOG2-scaled folded frames [E (n_fft/2) | O (n_fft/2)], reflect padding (center=True), T = L/hop + 1.
 *   acx_frontend_folded: w_hi / w_lo (ceil(n_chunks/2)*256, n_fft/2) fp16 pairs, per pair of 64-bin chunks the rows
 *     [re chunk 2p | re chunk 2p+1 | im chunk 2p | im chunk 2p+1] (engine.fold_dft_weights); mel_* / bn_* / out as below. */
ACX_API int acx_frame_fold(const float* wave, void* f_hi, void* f_lo, int B, int L, int T, int n_fft, int hop, void* stream);
ACX_API int acx_frame_fold_pcm16(const int16_t* pcm, void* f_hi, void* f_lo, int B, int L, int T, int n_fft, int hop, void* stream);
ACX_API int acx_frontend_folded(const void* f_hi, const void* f_lo, const void* w_hi, const void* w_lo, const void* mel_hi,
                        const void* mel_lo, int n_chunks, const float* bn_scale, const float* bn_shift, float* out,
                        int B, int T, int n_fft, int n_mels, void* stream);

ACX_API int acx_frontend_fused(const void* hi, const void* lo, int ld_pad, const void* dft_hi, const void* dft_lo,
                       const void* mel_hi, const void* mel_lo, int n_chunks, const float* bn_scale,
                       const float* bn_shift, float* out, int B, int T, int n_fft, int hop, int n_mels,
                       void* stream);

/* ---- stem: Conv2d(1,96,4x4,s4,pad=(4,0)) + channels_first LayerNorm (CX:688-691, CX:227) ---- */
/* logmel (B, T, 224) fp32 -> out (B, H0, 56, 96) act_dtype, H0 = (T+4)/4 + 1.
 * w (16, 96) fp32 = stem weight transposed to (ky*4+kx, cout). */
ACX_API int acx_stem(const float* logmel, const float* w, const float* bias, const float* ln_w, const float* ln_b,
             void* out, int B, int T, int n_mels, int act_dtype, void* stream);
/* bf16 mode, same stem writing the group-planar layout [12][Mp][8] (Mp = B*H0*56 rounded up to 128) directly */
ACX_API int acx_stem_gp(const float* logmel, const float* w, const float* bias, const float* ln_w, const float* ln_b,
                void* out, int B, int T, int n_mels, void* stream);

/* ---- Block part 1: depthwise 7x7 (pad 3, bias) + channels-last LayerNorm eps 1e-6 (CX:76-78) - */
/* x (B,H,W,C) -> y (B,H,W,C); w (49, C) act_dtype (dwconv weight transposed), W % 7 == 0. */
ACX_API int acx_dwconv_ln(const void* x, const void* w, const float* bias, const float* ln_w, const float* ln_b,
                  void* y, int B, int H, int W, int C, int act_dtype, void* stream);

/* ---- Block part 1 on the tensor cores (bf16 mode): depthwise 7x7 (pad 3) + bias (CX:76) as banded-Toeplitz
 *      tcgen05 GEMMs, then the channels-last LayerNorm (CX:78) as its own pass. -------------------------------- */
/* x (B,H,W,C) bf16 -> v (B,H,W,C) bf16 = conv + bias, NOT normalised; w (49, C) bf16; W in {56,28,14,7}, C % 8 == 0;
 * out of place. */
ACX_API int acx_dwconv_tc(const void* x, const void* w, const float* bias, void* v, int B, int H, int W, int C,
                  void* stream);
/* rows of C bf16 values: out = LayerNorm(in) * ln_w + ln_b, eps 1e-6, fp32 statistics; in == out allowed. */
ACX_API int acx_layernorm_rows(const void* in, const float* ln_w, const float* ln_b, void* out, long long M, int C,
                       void* stream);

/* Group-planar hand-off layout of stages 0 / 1 in bf16 mode: [C/8][Mp][8] (M = B*H*W pixels, each 16-byte group of 8
 * channels is a plane; the plane stride Mp is M rounded up to a multiple of 128 rows -- buffers hold C * Mp elements) -- the tensor-core depthwise conv then moves whole cache lines.  acx_gp_transpose converts
 * (M, C) row-major <-> planar (to_gp = 1 / 0); acx_dwconv_tc_gp is acx_dwconv_tc on planar x / v (W in {56, 28}). */
ACX_API int acx_dwconv_tc_gp(const void* x, const void* w, const float* bias, void* v, int B, int H, int W, int C,
                     void* stream);
ACX_API int acx_gp_transpose(const void* in, void* out, long long M, int C, int to_gp, void* stream);
/* stats[row] = (rstd, -mean * rstd) of the C channels of each row of a group-planar tensor (LayerNorm eps 1e-6) */
ACX_API int acx_gp_row_stats(const void* v, float* stats, long long M, int C, void* stream);

/* ---- downsample prologue: channels_first LayerNorm + 2x2/s2 patch gather (CX:231-234) ------- */
/* x (B,H,W,C) -> a (B*(H/2)*(W/2), 4C) with k = (dy*2+dx)*C + c  (the GEMM A operand). */
ACX_API int acx_ln_patchify(const void* x, const float* ln_w, const float* ln_b, void* a, int B, int H, int W, int C,
                    int act_dtype, void* stream);
/* same, x group-planar [C/8][B*H*W][8] bf16 (C = 96 / 192); `a` row-major as above */
ACX_API int acx_ln_patchify_gp(const void* x, const float* ln_w, const float* ln_b, void* a, int B, int H, int W, int C,
                       void* stream);

/* ---- the whole downsample layer as one implicit GEMM (CX:230-235: LayerNorm(channels_first) -> Conv2d(k2, s2)) ----
 * x group-planar bf16 [C/8][Mp][8] (Mp = B*H*W rounded up to 128); the LayerNorm'd 2x2 patches are formed in shared memory
 * as the tensor-core A operand (no patch matrix in HBM).  w: (2C, 4C) bf16, k = ((dy * C/8 + g) * 2 + dx) * 8 + c8 for
 * input channel 8 g + c8 at patch position (dy, dx).  out: (B*(H/2)*(W/2), 2C) bf16 row-major, or group-planar
 * [2C/8][Mp_out][8] when out_gp.  C = 96 / 192 / 384, W even (an odd last row of H is dropped like the conv does). */
ACX_API int acx_downsample_fused_gp(const void* x, const float* ln_w, const float* ln_b, const void* w, const float* bias,
                            void* out, int B, int H, int W, int C, int out_gp, void* stream);

/* ---- GEMMs: out[M,N] = epi(A[M,K] . W[N,K]^T)  (nn.Linear / conv-as-GEMM weight layout) ------ */
/* bf16 operands, fp32 accumulation in TMEM (tcgen05.mma, TMA-fed).  K % 8 == 0, N % 32 == 0. */
ACX_API int acx_gemm_bf16(const void* A, const void* W, void* out, int M, int N, int K, int epilogue,
                  const float* bias, const float* gamma, const void* resid, void* stream);
/* out = A . W^T + bias written group-planar, [N/8][Mp][8] with Mp = M rounded up to 128 (bias epilogue only) */
ACX_API int acx_gemm_bf16_gp_out(const void* A, const void* W, void* out, int M, int N, int K, const float* bias,
                         void* stream);
/* The two GEMMs of a Block MLP on group-planar activations (stage 2, whose MLP is not the fused kernel):
 *   pw1: hid (M, N = 4C) row-major = GELU(LN(v) . W1^T + b1), v planar [K/8][Mp][8], LayerNorm folded: w1f = bf16(W1 ln_w),
 *        b1f = b1 + W1 ln_b, ln_s[j] = sum_k w1f[j, k], stats = acx_gp_row_stats(v);
 *   pw2: x (planar [N/8][Mp][8], in place) += gamma * (hid . W2^T + b2). */
ACX_API int acx_gemm_bf16_pw1_gp(const void* v_gp, const void* w1f, void* hid, int M, int N, int K, const float* b1f,
                         const float* stats, const float* ln_s, void* stream);
ACX_API int acx_gemm_bf16_pw2_gp(const void* hid, const void* w2, void* x_gp, int M, int N, int K, const float* b2,
                         const float* gamma, void* stream);
/* fp32 SIMT GEMM of the fp32-accurate path.  Row m of A starts at
 * A + (m / rows_per_batch) * batch_stride + (m % rows_per_batch) * row_stride (elements), which
 * also expresses the overlapping STFT frames (row_stride = hop). */
ACX_API int acx_gemm_f32(const float* A, long long batch_stride, int rows_per_batch, int row_stride, const float* W,
                 float* out, int ldo, int M, int N, int K, int epilogue, const float* bias,
                 const float* gamma, const float* resid, void* stream);

/* ---- Block part 2, fused: pwconv1 -> GELU -> pwconv2 -> gamma -> +residual (CX:79-86) -------- */
/* y (M,C) bf16 LN output; x (M,C) bf16 residual stream, updated IN PLACE.
 * w1 (4C,C), w2 (C,4C) bf16.  The 4C hidden tile lives in TMEM/SMEM only.  C in {96,192}. */
ACX_API int acx_mlp_fused(const void* y, void* x, const void* w1, const float* b1, const void* w2, const float* b2,
                  const float* gamma, int M, int C, void* stream);
/* Same with the Block's channels-last LayerNorm (CX:78, eps 1e-6) applied to the operand tile in shared memory:
 * v (M, C) bf16 is the RAW depthwise-conv output of acx_dwconv_tc; no normalised copy ever exists in HBM. */
ACX_API int acx_mlp_fused_ln(const void* v, void* x, const float* ln_w, const float* ln_b, const void* w1,
                     const float* b1, const void* w2, const float* b2, const float* gamma, int M, int C,
                     void* stream);
/* Group-planar variant: v and x are [C/8][Mp][8] bf16 (each 16-byte group of 8 channels of all rows is a plane, plane
 * stride Mp = M rounded up to 128), the hand-off layout of acx_dwconv_tc_gp.  Three LayerNorm modes:
 *   ln_w = ln_b = ln_s = NULL   v is already normalised;
 *   ln_w, ln_b given            the LayerNorm is applied to the operand tile in shared memory;
 *   ln_s given (ln_w/ln_b NULL) FOLDED: w1 = bf16(W1 diag(ln_w)), b1 = b1 + W1 ln_b, ln_s[j] = sum_c w1[j, c]; the kernel
 *                               computes per-row statistics only and applies the LayerNorm as a rank-1 correction
 *                               rstd (G - mean s) + b1 in the GELU epilogue. */
ACX_API int acx_mlp_fused_gp(const void* v, void* x, const float* ln_w, const float* ln_b, const float* ln_s,
                     const void* w1, const float* b1, const void* w2, const float* b2, const float* gamma, int M, int C,
                     void* stream);

/* ---- tail: mean over mel, max_t + mean_t, LayerNorm(768), fc 768->527, sigmoid (CX:279-285, 321-325) */
/* x (B,H,W,C) act_dtype -> scene (B,C) fp32 [post-LN], logits (B,n_cls), probs (B,n_cls).
 * pooled (B,C) fp32 is caller-provided scratch (the pre-LayerNorm pooled vector). */
ACX_API int acx_head(const void* x, const float* ln_w, const float* ln_b, const float* fc_w, const float* fc_b,
             float* pooled, float* scene, float* logits, float* probs, int B, int H, int W, int C, int n_cls,
             int act_dtype, void* stream);

/* x (B,H,W,C) act_dtype -> out (B,C,H,W) fp32: the layout forward_frame_embeddings returns (CX:399-402). */
ACX_API int acx_nhwc_to_nchw_f32(const void* x, float* out, int B, int H, int W, int C, int act_dtype, void* stream);

/* ---- ragged batches: clips of different lengths in one launch sequence -------------------------------------------------
 * Clip b sits in row b of a canvas sized for the longest clip; every size argument is the CANVAS size.  `valid` (device,
 * B int32 entries) gives each clip's own extent in the unit the kernel bounds:
 *   acx_wave_prep_ragged, acx_frame_fold_ragged   samples L_b (the input rows are ld_wave apart, ld_wave >= L)
 *   acx_stem_ragged, acx_stem_gp_ragged           frames  T_b = L_b / hop + 1
 *   acx_dwconv_*_ragged                           rows    h_b of the stage (h0_b = (T_b + 4) / 4 + 1, h(s+1)_b = h(s)_b / 2)
 *   acx_head_ragged, acx_nhwc_to_nchw_f32_ragged  rows    h3_b of the last stage
 * A clip's rows past its extent are never read: the prep kernels reflect at L_b and write zeros past L_b + n_fft, the
 * convolutions read those rows as their own zero padding, the head pools over h3_b rows, and the frame transpose writes
 * zeros there.  Rows below the extent therefore equal a run of the clip alone at its own length, bit for bit; rows past
 * it hold values without meaning.  The kernels clamp each entry to the canvas (and to what their indexing needs: > n_fft/2
 * samples for the prep kernels, >= 1 row for the head), so no value can make them access memory outside their buffers;
 * whether the values are right (L_b > n_fft/2, h3_b >= 1, entries consistent with each other) is for the caller to check.
 * A null `valid` returns ACX_ERR_ARG. */
ACX_API int acx_wave_prep_ragged(const float* wave, void* hi, void* lo, int B, int L, int n_fft, int ld_pad, int act_dtype,
                                 int ld_wave, const int32_t* valid, void* stream);
ACX_API int acx_frame_fold_ragged(const float* wave, void* f_hi, void* f_lo, int B, int L, int T, int n_fft, int hop,
                                  int ld_wave, const int32_t* valid, void* stream);
ACX_API int acx_stem_ragged(const float* logmel, const float* w, const float* bias, const float* ln_w, const float* ln_b,
                            void* out, int B, int T, int n_mels, int act_dtype, const int32_t* valid, void* stream);
ACX_API int acx_stem_gp_ragged(const float* logmel, const float* w, const float* bias, const float* ln_w, const float* ln_b,
                               void* out, int B, int T, int n_mels, const int32_t* valid, void* stream);
ACX_API int acx_dwconv_tc_ragged(const void* x, const void* w, const float* bias, void* v, int B, int H, int W, int C,
                                 const int32_t* valid, void* stream);
ACX_API int acx_dwconv_tc_gp_ragged(const void* x, const void* w, const float* bias, void* v, int B, int H, int W, int C,
                                    const int32_t* valid, void* stream);
ACX_API int acx_dwconv_ln_ragged(const void* x, const void* w, const float* bias, const float* ln_w, const float* ln_b,
                                 void* y, int B, int H, int W, int C, int act_dtype, const int32_t* valid, void* stream);
ACX_API int acx_head_ragged(const void* x, const float* ln_w, const float* ln_b, const float* fc_w, const float* fc_b,
                            float* pooled, float* scene, float* logits, float* probs, int B, int H, int W, int C, int n_cls,
                            int act_dtype, const int32_t* valid, void* stream);
ACX_API int acx_nhwc_to_nchw_f32_ragged(const void* x, float* out, int B, int H, int W, int C, int act_dtype,
                                        const int32_t* valid, void* stream);

/* ---- windows of a long recording: prep kernels that read each window in place --------------------------------------
 * Row b of the batch is the window that starts offsets[b] samples into ONE recording `rec` of rec_len samples (fp32, or
 * int16 PCM converted x / 32767. like acx_wave_prep_pcm16).  Windows may overlap and offsets are 64-bit, so a recording
 * may be longer than 2^31 samples.  Every size argument is the CANVAS size, as for the ragged entry points; the outputs
 * are exactly those of acx_wave_prep / acx_frame_fold on the batch of copied windows, so every later kernel is unchanged.
 *   valid == NULL   every window has L samples;
 *   valid != NULL   row 0 of the chunk's ragged bound table (B int32 entries): window b has its own L_b samples and is
 *                   reflected at its own end, as in acx_wave_prep_ragged; the later kernels then run their _ragged forms.
 * A window never reads a sample outside [offsets[b], offsets[b] + L_b).  Each length is clamped to rec_len (and, with
 * valid, to [n_fft/2 + 1, L]), each offset to [0, rec_len - length], so no value can make the kernels read outside the
 * recording; whether the values are right is for the caller to check.  A null rec or offsets, rec_len <= n_fft/2 or
 * B < 1 returns ACX_ERR_ARG. */
ACX_API int acx_wave_prep_windows(const float* rec, long long rec_len, const long long* offsets, const int32_t* valid,
                                  void* hi, void* lo, int B, int L, int n_fft, int ld_pad, int act_dtype, void* stream);
ACX_API int acx_wave_prep_pcm16_windows(const int16_t* rec, long long rec_len, const long long* offsets,
                                        const int32_t* valid, void* hi, void* lo, int B, int L, int n_fft, int ld_pad,
                                        int act_dtype, void* stream);
ACX_API int acx_frame_fold_windows(const float* rec, long long rec_len, const long long* offsets, const int32_t* valid,
                                   void* f_hi, void* f_lo, int B, int L, int T, int n_fft, int hop, void* stream);
ACX_API int acx_frame_fold_pcm16_windows(const int16_t* rec, long long rec_len, const long long* offsets,
                                         const int32_t* valid, void* f_hi, void* f_lo, int B, int L, int T, int n_fft,
                                         int hop, void* stream);

/* ---- next row (f4): demo preprocessing, reference demo_convnext.py:52-67 --------------------- */
/* torchaudio.functional.resample (sinc_interp_hann polyphase FIR, demo_convnext.py:53-59) fused with the demo's
 * constant pad / crop to a fixed clip length (demo_convnext.py:61-67):
 *   out[b, f*newf + p] = sum_{k<K} taps[k*newf + p] * x[b, f*orig + k - width]      (x = 0 outside [0, L_in))
 * for output index i < ceil(newf * L_in / orig), zero from there to n_out, cropped at n_out.
 * orig/newf are the rates divided by their gcd, K = 2*width + orig; taps (K, newf) fp32 is the TRANSPOSED
 * torchaudio kernel, built on the host (preprocess.sinc_resample_taps).  x (B, ld_in), out (B, ld_out). */
ACX_API int acx_resample_fit(const float* x, int ld_in, const float* taps, float* out, int ld_out, int B, int L_in,
                     int orig, int newf, int width, int n_out, void* stream);

/* ---- any sample rate: recordings of any lengths resampled in one launch per rate ---------------------------------------
 * x holds S segments packed in one buffer of x_len samples (fp32, or int16 PCM converted x / 32767. with a correctly
 * rounded division, like acx_wave_prep_pcm16); out is one fp32 buffer of out_len samples.  seg is a DEVICE (S, 4) int64
 * table, row s = (in_off, in_len, out_off, out_len) in samples of x and out.  Output j < out_len of segment s is
 *   sum_{k<K} taps[k*newf + p] * v(f*orig - width + k),   f = j / newf, p = j % newf,
 * accumulated with fmaf in k order, where v(i) = x[in_off + i] for 0 <= i < in_len and ZERO outside the segment: a
 * segment never reads its neighbours' samples.  So each segment equals acx_resample_fit of that segment alone with
 * n_out = ceil(newf * in_len / orig), bit for bit, and out_len is normally that ceil.  Indices are 64-bit, so a segment
 * may exceed 2^31 samples.  Each entry is clamped to x_len / out_len, so no table value makes the kernel read or write
 * outside its buffers; whether the values are right is for the caller to check.
 * Work distribution: one block per tile of tile_frames frames x (taps' phases / phase_groups) phases of one segment.
 * Segment s owns ceil(ceil(out_len_s / newf) / tile_frames) * phase_groups tiles, starting at tile_start[s] (DEVICE (S,)
 * int64, non-decreasing, tile_start[0] = 0); n_tiles is the total.  acx_resample_segments_tiling gives tile_frames and
 * phase_groups for a rate pair (host call, no launch), and returns ACX_ERR_UNSUPPORTED when the tile's taps and input span
 * exceed shared memory (about 58 000 floats: K * 4 * phase warps + (tile_frames - 1) * orig + K; 8 to 192 kHz -> 32 kHz
 * and 11.025 / 22.05 / 44.1 / 88.2 kHz all fit).
 * A null pointer, S < 1, x_len < 1, out_len < 1, n_tiles outside [1, 2^31) or a rate or width <= 0 returns ACX_ERR_ARG
 * before any launch. */
ACX_API int acx_resample_segments_tiling(int orig, int newf, int width, int* tile_frames_host, int* phase_groups_host);
ACX_API int acx_resample_segments(const float* x, long long x_len, const long long* seg, int S,
                                  const long long* tile_start, long long n_tiles, const float* taps, int orig, int newf,
                                  int width, float* out, long long out_len, void* stream);
ACX_API int acx_resample_segments_pcm16(const int16_t* x, long long x_len, const long long* seg, int S,
                                        const long long* tile_start, long long n_tiles, const float* taps, int orig,
                                        int newf, int width, float* out, long long out_len, void* stream);

/* ---- live streams: per-stream rings in one fp32 buffer ---------------------------------------------------------------
 * acx_stream_append(_pcm16) scatters one push's chunks, packed end to end in src (src_len samples; fp32, or int16 PCM
 * converted x / 32767. with a correctly rounded division), into the streams' rings in ONE launch.  table is a DEVICE
 * (S, 6) int64 table, row s = (src_off, n, ring_base, cap, pos, mirror), rows in src order: sample i < n of chunk s goes
 * to ring[ring_base + (pos + i) mod cap], and also to ring[ring_base + cap + (pos + i) mod cap] when that slot is below
 * `mirror` (so a window of up to `mirror` samples starting anywhere in the ring is contiguous).  Each entry is clamped
 * (src_off to [0, src_len], n <= cap, pos reduced mod cap, mirror <= cap, [ring_base, ring_base + cap + mirror) inside
 * ring_len): no table value makes the kernel write outside its row's region.  A null pointer, S < 1, src_len outside [1, 2^39) or ring_len < 1 returns
 * ACX_ERR_ARG before any launch. */
ACX_API int acx_stream_append(const float* src, long long src_len, const long long* table, int S, float* ring,
                              long long ring_len, void* stream);
ACX_API int acx_stream_append_pcm16(const int16_t* src, long long src_len, const long long* table, int S, float* ring,
                                    long long ring_len, void* stream);

/* acx_resample_stream: the streaming form of acx_resample_segments (same taps, tiling, tile prefix and argument checks;
 * fp32 input only).  table is a DEVICE (S, 8) int64 table, row s = (in_base, in_cap, in_end, f0, n_out, out_base,
 * out_cap, out_mirror) for one stream: its input sample idx is x[in_base + idx mod in_cap] for 0 <= idx < in_end and
 * zero otherwise, and the row computes the n_out outputs j = f0 * newf + jl (jl < n_out; f0 a 64-bit stream frame) with
 * the same fmaf chain as acx_resample_segments.  Output j goes to out[out_base + j mod out_cap], and also to
 * out[out_base + out_cap + j mod out_cap] when that slot is below out_mirror.  So outputs computed piece by piece equal
 * acx_resample_segments of the whole stream bit for bit, as long as the ring still holds every sample a frame reads
 * (the caller's invariant).  Tiles are counted on n_out as segments count them on out_len.  Entries are clamped to
 * x_len / out_len like the segments' are (in_cap and out_cap >= 1 or the row is skipped, out_mirror <= out_cap, f0 to
 * [0, 2^62 / max(orig, newf)] so that no index overflows): no table value makes the kernel read or write outside its
 * row's regions.  x and out may be one buffer when the regions do not overlap. */
ACX_API int acx_resample_stream(const float* x, long long x_len, const long long* table, int S,
                                const long long* tile_start, long long n_tiles, const float* taps, int orig, int newf,
                                int width, float* out, long long out_len, void* stream);

/* ---- sound event detection: window rows -> activity bins -> timed events (527 classes) --------------------------------
 * acx_window_activity: probs is (p_rows, 527) fp32 clipwise rows (a forward_windows result, or a ring of a stream's
 * recent rows); table is a DEVICE (M, 4) int64 table, one row per output bin, row m = (row_first, n, ring_base, ring_cap).
 * Row t < n of bin m is probs[ring_base + (row_first + t) mod ring_cap], and
 *   act[m, c] = (sum over t of those rows' column c) / n,
 * the sum taken with plain fp32 adds in t order starting from the first row, the division correctly rounded (act is
 * (M, 527) fp32).  A whole recording uses ring_base = 0, ring_cap = p_rows.  Every entry is clamped (ring_cap to
 * [1, p_rows], ring_base to [0, p_rows - ring_cap], n to [0, ring_cap], row_first reduced mod ring_cap): no table value
 * reads outside probs; a bin with n = 0 reads nothing and is NaN.  A null pointer, p_rows < 1, M < 1 or M > 2^40 / 527
 * returns ACX_ERR_ARG before any launch. */
ACX_API int acx_window_activity(const float* probs, long long p_rows, const long long* table, long long M, float* act,
                                void* stream);

/* acx_detect_events: one thread per (sequence, class) track walks the sequence's new bins through the hysteresis state
 * machine (open at act >= on[c], stay open while act >= off[c], end at the first bin where !(act >= off[c]); consecutive
 * events merge when next onset - previous offset < merge_gap; an event is kept when offset - onset >= min_duration).  seq
 * is a DEVICE (S, 6) int64 table, row s = (recording, row0, n_bins, j0, limit, close): the sequence's new bins are act
 * rows row0 .. row0 + n_bins - 1 with bin indices j0 .. j0 + n_bins - 1, bin j spans [j resolution, min((j + 1)
 * resolution, limit)), and close != 0 ends the sequence.  state ((3, S * 527) int64: phase 0 idle / 1 open / 2 ended but
 * may merge, onset bin, last bin) and state_peak ((S * 527) fp32) carry each track from call to call; zeros are a fresh
 * track.  An event is emitted once no later bin can change it: at close, or once the next bin's start minus its offset
 * reaches merge_gap.  phase 0 writes the number of events each track emits to slots[s * 527 + c] and changes nothing
 * else; the caller turns the counts into their exclusive prefix in place, and phase 1 writes the events from those slots
 * and stores the state: out is (4, E) int64 rows (recording, class, onset, offset) in samples and out_peak (E,) fp32 the
 * max activity over the event's bins, ordered (sequence, class, onset).  row0 and n_bins are clamped to act_rows, and no
 * event is written outside [0, E).  A null pointer (act may be null with act_rows = 0, out / out_peak with E = 0 or in
 * phase 0), S outside [1, 2^30 / 527], act_rows outside [0, 2^40 / 527], E < 0, resolution < 1, merge_gap < 0,
 * min_duration < 0 or a phase other than 0 / 1 returns ACX_ERR_ARG before any launch. */
ACX_API int acx_detect_events(const float* act, long long act_rows, const long long* seq, int S,
                              const float* on_threshold, const float* off_threshold, long long resolution,
                              long long merge_gap, long long min_duration, long long* state, float* state_peak,
                              long long* slots, int phase, long long* out, float* out_peak, long long E, void* stream);

/* ---- query by example: exact cosine search over embedding rows -------------------------------------------------------
 * acx_row_norms: out[r] = sqrt(sum_i x[r, i]^2) (fp64) for the (rows, d) fp32 rows x, the sum taken in fp64 in i order
 * from 0.0.  A null pointer, rows outside [1, 2^40] or d < 1 returns ACX_ERR_ARG before any launch. */
ACX_API int acx_row_norms(const float* x, long long rows, int d, double* out, void* stream);

/* acx_cosine_scores: scores (Q, N) fp32, row-major, scores[q, n] = float32(dot / (query_norms[q] * key_norms[n])), where
 * dot = sum_i queries[q, i] * keys[n, i] is the fp64 fma chain over i = 0 .. d-1 in order from 0.0 (every product of two
 * fp32 values is exact in fp64, so it equals the plain fp64 sum), the product and quotient are rounded once each in fp64
 * and the conversion rounds to nearest even; a NaN result is stored as 0x7fc00000.  queries (Q, d) and keys (N, d) fp32
 * are row-major, the norms are acx_row_norms results.  Indices are 64-bit: Q * N may exceed 2^31.  A null pointer, Q
 * outside [1, 65535 * 64], N outside [1, 2^31 - 1] or d < 1 returns ACX_ERR_ARG before any launch. */
ACX_API int acx_cosine_scores(const float* queries, const double* query_norms, long long Q, const float* keys,
                              const double* key_norms, long long N, int d, float* scores, void* stream);

/* acx_search_topk: for every row q of scores ((Q, N) fp32, an acx_cosine_scores result), the top k' = min(k, eligible)
 * rows under the order "a beats b when score_a > score_b, or the scores are equal and a < b" (-0.0 equals +0.0; NaN ranks
 * below every number and NaNs tie).  Row w is eligible when it beats every row j != w in [lo_w, hi_w), (lo_w, hi_w) = row
 * w of ranges, a DEVICE (N, 2) int64 table, each entry clamped to [0, N]; ranges = null makes every row eligible.
 * out_score (Q, k) fp32 and out_index (Q, k) int64 receive the hits best first; slots k' .. k-1 get score NaN
 * (0x7fc00000) and index -1.  workspace is DEVICE scratch of acx_search_topk_workspace(Q, N) bytes (a host query, no
 * launch).  Two launches, no allocation and no synchronisation.  A null pointer (ranges excepted), Q or N outside
 * [1, 2^31 - 1] or k outside [1, 1024] returns ACX_ERR_ARG before any launch. */
ACX_API int acx_search_topk_workspace(long long Q, long long N, long long* bytes_host);
ACX_API int acx_search_topk(const float* scores, long long Q, long long N, const long long* ranges, int k,
                            float* out_score, long long* out_index, void* workspace, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ACX_H_ */
