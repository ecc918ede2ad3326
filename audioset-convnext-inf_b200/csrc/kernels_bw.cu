// CUDA-core / bandwidth kernels of the hot path (channels-last, H = time, W = mel):
//   wave_prep        reflect pad + fp32 -> scaled fp16 hi/lo split            (torchlibrosa STFT.forward pad)
//   power_mel_log    re^2+im^2 -> banded mel -> 10 log10 -> bn0        (fp32-accurate path)
//   stem             4x4/s4 patchify conv + LayerNorm(96)              (CX:688-691, CX:227)
//   dwconv_ln        depthwise 7x7 + channels-last LayerNorm           (CX:76-78)
//   ln_patchify      channels_first LayerNorm + 2x2 patch gather       (CX:231-234)
//   head             mel-mean, time max+mean, LayerNorm, fc, sigmoid   (CX:279-285, CX:321-325)
//   nhwc_to_nchw     frame-embedding layout                            (CX:399-402)
// "CX" = reference src/audioset_convnext_inf/pytorch/convnext.py.
#include <type_traits>

#include "common.cuh"

namespace acx {

// =============================================================================================
// wave_prep
// =============================================================================================
// TIn = float (waveform) or int16_t (PCM as stored in the AudioSet HDF5 files; converted exactly like the reference's
// int16_to_float32, utils/utilities.py:226-227: x / 32767. -- a true division, not a reciprocal multiply).
__device__ __forceinline__ float load_sample(const float* p) { return __ldg(p); }
__device__ __forceinline__ float load_sample(const int16_t* p) { return __fdiv_rn((float)__ldg(p), 32767.0f); }

// RAG: row b is a clip of valid[b] samples (clamped to [pad + 1, L]) at row pitch ld_wave; it is reflected at its own end
// and zero past it, exactly like a run at that length.  Samples past valid[b] are never read.
// WIN: row b is the window that starts offsets[b] samples into ONE recording of rec_len samples (windows may overlap); it
// has L samples, or with RAG its own valid[b].  Offsets are 64-bit.  The length is clamped to rec_len and the offset to
// [0, rec_len - length], so no table value can make the kernel read outside the recording.
template <bool kSplit, typename TIn, bool RAG = false, bool WIN = false>
__global__ void wave_prep_kernel(const TIn* __restrict__ wave, void* __restrict__ hi_, void* __restrict__ lo_,
                                 int L, int pad, int ld_pad, int ld_wave, const int32_t* __restrict__ valid,
                                 const long long* __restrict__ offsets = nullptr, long long rec_len = 0) {
  // 4 consecutive output samples per thread (ld_pad % 8 == 0): 8-byte bf16 / 16-byte fp32 stores
  const int b = blockIdx.y;
  const int j0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (j0 >= ld_pad) return;
  if (RAG) L = min(max(__ldg(valid + b), pad + 1), L);
  const TIn* win = wave;
  if (WIN) {
    L = (int)min((long long)L, rec_len);
    win = wave + min(max(__ldg(offsets + b), 0LL), rec_len - L);
  }
  float v[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int j = j0 + i;
    v[i] = 0.f;
    if (j < L + 2 * pad) {
      int s = j - pad;
      if (s < 0) s = -s;                       // reflect (edge sample not repeated)
      if (s >= L) s = 2 * (L - 1) - s;
      v[i] = load_sample(WIN ? win + s : wave + (size_t)b * (RAG ? ld_wave : L) + s);
    }
  }
  const size_t o = (size_t)b * ld_pad + j0;
  if (kSplit) {
    // fp16 hi / lo of 2^ACX_FE_SCALE_LOG2 * x (see acx.h): 22 mantissa bits for the tensor-core DFT
    constexpr float kScale = (float)(1 << ACX_FE_SCALE_LOG2);
    uint32_t h[2], l[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const float s0 = v[2 * i] * kScale, s1 = v[2 * i + 1] * kScale;
      const __half2 hh = __floats2half2_rn(s0, s1);
      const float2 hf = __half22float2(hh);
      const __half2 ll = __floats2half2_rn(s0 - hf.x, s1 - hf.y);
      h[i] = *reinterpret_cast<const uint32_t*>(&hh);
      l[i] = *reinterpret_cast<const uint32_t*>(&ll);
    }
    *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(hi_) + o) = make_uint2(h[0], h[1]);
    *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(lo_) + o) = make_uint2(l[0], l[1]);
  } else {
    *reinterpret_cast<float4*>(reinterpret_cast<float*>(hi_) + o) = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// =============================================================================================
// power -> mel -> log -> bn0 (fp32-accurate path; spectrogram materialised by the SIMT GEMM)
// =============================================================================================
__global__ void power_mel_log_kernel(const float* __restrict__ spec, int ld_spec, int n_bins,
                                     const float* __restrict__ melT, const int32_t* __restrict__ mel_lo,
                                     const int32_t* __restrict__ mel_hi, const float* __restrict__ bn_scale,
                                     const float* __restrict__ bn_shift, float* __restrict__ out, int rows,
                                     int n_mels) {
  extern __shared__ float p[];
  const int r = blockIdx.x;
  const float* s = spec + (size_t)r * ld_spec;
  for (int k = threadIdx.x; k < n_bins; k += blockDim.x) {
    const float re = s[k], im = s[n_bins + k];
    p[k] = re * re + im * im;
  }
  __syncthreads();
  for (int m = threadIdx.x; m < n_mels; m += blockDim.x) {
    const int lo = mel_lo[m], hi = mel_hi[m];
    const float* w = melT + (size_t)m * n_bins;
    float acc = 0.f;
    for (int k = lo; k < hi; ++k) acc = fmaf(p[k], w[k], acc);
    const float db = 10.0f * log10f(fmaxf(acc, 1e-10f));
    out[(size_t)r * n_mels + m] = db * bn_scale[m] + bn_shift[m];
  }
}

// =============================================================================================
// stem: 4x4 stride-4 conv over (T, 224) with 4 rows of zero padding in time, then LayerNorm(96)
// (reference convnext.py:688-691 + :227).  One THREAD per output pixel, all 96 channels in registers:
//  * the 16 patch values are four coalesced float4 loads (consecutive pixels = consecutive 16 B);
//  * the (16, 96) taps sit in smem and are read with warp-uniform LDS.128 (broadcast), 1 per 4 channels, and
//    applied with packed fp32x2 FMAs;
//  * LayerNorm statistics need no cross-thread traffic at all;
//  * the warp's 32 x 96 outputs (contiguous in HBM) are transposed through padded smem and stored coalesced.
// =============================================================================================
// RAG: clip b has valid[b] frames (clamped to [0, Tn]); later rows are read as the conv's zero padding.
template <typename T, bool RAG = false>
__global__ void __launch_bounds__(128) stem_kernel(const float* __restrict__ logmel, const float* __restrict__ w,
                                                   const float* __restrict__ bias, const float* __restrict__ ln_w,
                                                   const float* __restrict__ ln_b, T* __restrict__ out, int B,
                                                   int Tn, int n_mels, int H0, int W0, const int32_t* __restrict__ valid) {
  constexpr int CO = 96;
  constexpr int ROW_BYTES = CO * (int)sizeof(T);       // 192 (bf16) / 384 (fp32)
  constexpr int ROW_PITCH = ROW_BYTES + 16;            // +16 B: conflict-free 16-byte row writes
  extern __shared__ __align__(16) uint8_t ssm[];
  float* sw = reinterpret_cast<float*>(ssm);           // [16][96] taps, then bias / ln_w / ln_b [3][96]
  uint8_t* stile = ssm + (16 + 3) * CO * 4 + (threadIdx.x >> 5) * 32 * ROW_PITCH;
  for (int i = threadIdx.x; i < 16 * CO; i += blockDim.x) sw[i] = w[i];
  for (int i = threadIdx.x; i < CO; i += blockDim.x) {
    sw[16 * CO + i] = bias[i];
    sw[17 * CO + i] = ln_w[i];
    sw[18 * CO + i] = ln_b[i];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long total = (long long)B * H0 * W0;
  const long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long warp_pix0 = pix - lane;
  const bool ok = pix < total;
  float xin[16];
  {
    const long long pp = ok ? pix : 0;
    const int ox = (int)(pp % W0);
    const int oy = (int)((pp / W0) % H0);
    const int b = (int)(pp / ((long long)W0 * H0));
    const int Tb = RAG ? min(max(__ldg(valid + b), 0), Tn) : Tn;
#pragma unroll
    for (int ky = 0; ky < 4; ++ky) {
      const int t = oy * 4 - 4 + ky;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ok && t >= 0 && t < Tb) v = __ldg(reinterpret_cast<const float4*>(logmel + ((size_t)b * Tn + t) * n_mels + ox * 4));
      xin[ky * 4 + 0] = v.x;
      xin[ky * 4 + 1] = v.y;
      xin[ky * 4 + 2] = v.z;
      xin[ky * 4 + 3] = v.w;
    }
  }
  float2 acc[CO / 2];
#pragma unroll
  for (int c = 0; c < CO / 2; c += 2) {
    const float4 b4 = *reinterpret_cast<const float4*>(sw + 16 * CO + 2 * c);
    acc[c] = make_float2(b4.x, b4.y);
    acc[c + 1] = make_float2(b4.z, b4.w);
  }
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const float2 xv = make_float2(xin[k], xin[k]);
#pragma unroll
    for (int c = 0; c < CO / 2; c += 2) {
      const float4 w4 = *reinterpret_cast<const float4*>(sw + k * CO + 2 * c);   // warp-uniform -> broadcast
      acc[c] = __ffma2_rn(xv, make_float2(w4.x, w4.y), acc[c]);
      acc[c + 1] = __ffma2_rn(xv, make_float2(w4.z, w4.w), acc[c + 1]);
    }
  }
  float sum = 0.f;
#pragma unroll
  for (int c = 0; c < CO / 2; ++c) sum += acc[c].x + acc[c].y;
  const float mean = sum * (1.0f / CO);
  float sq = 0.f;
#pragma unroll
  for (int c = 0; c < CO / 2; ++c) {
    acc[c].x -= mean;
    acc[c].y -= mean;
    sq = fmaf(acc[c].x, acc[c].x, sq);
    sq = fmaf(acc[c].y, acc[c].y, sq);
  }
  const float rstd = rsqrtf(sq * (1.0f / CO) + 1e-6f);
  // normalise, convert, and write this pixel's row into the warp tile
  uint8_t* myrow = stile + lane * ROW_PITCH;
#pragma unroll
  for (int c = 0; c < CO / 2; c += 2) {
    const float4 g4 = *reinterpret_cast<const float4*>(sw + 17 * CO + 2 * c);
    const float4 h4 = *reinterpret_cast<const float4*>(sw + 18 * CO + 2 * c);
    const float o0 = acc[c].x * rstd * g4.x + h4.x, o1 = acc[c].y * rstd * g4.y + h4.y;
    const float o2 = acc[c + 1].x * rstd * g4.z + h4.z, o3 = acc[c + 1].y * rstd * g4.w + h4.w;
    if (sizeof(T) == 2) {
      *reinterpret_cast<uint2*>(myrow + c * 4) = make_uint2(Pair<bf16>::pack(o0, o1), Pair<bf16>::pack(o2, o3));
    } else {
      *reinterpret_cast<float4*>(myrow + c * 8) = make_float4(o0, o1, o2, o3);
    }
  }
  __syncwarp();
  // coalesced copy-out: the warp's 32 rows are contiguous in global memory
  const long long n_valid = total - warp_pix0 < 32 ? total - warp_pix0 : 32;
  uint8_t* gdst = reinterpret_cast<uint8_t*>(out) + (size_t)warp_pix0 * ROW_BYTES;
  constexpr int PIECES = ROW_BYTES / 16;               // 16-byte pieces per row
  for (int i = lane; i < (int)n_valid * PIECES; i += 32) {
    const int r = i / PIECES, pc = i % PIECES;
    *reinterpret_cast<uint4*>(gdst + (size_t)r * ROW_BYTES + pc * 16) =
        *reinterpret_cast<const uint4*>(stile + r * ROW_PITCH + pc * 16);
  }
}

// =============================================================================================
// depthwise 7x7 + LayerNorm (reference convnext.py:76-78).
// Thread = one channel pair x a strip of 7 output pixels along W x R = 4 consecutive output rows.
//  * the two channels of a pair are processed by ONE packed fp32x2 FMA (FFMA2, new on sm_100);
//  * the R+6 input rows slide through registers: each row is loaded ONCE (13 channel-pair words, prefetched one
//    row ahead) and feeds up to 4 output rows -> 3.25 loads + 6.5 unpack ops per 98 FMAs;
//  * the 49 taps of every channel live in shared memory as fp32 pairs (one conflict-free LDS.64 per 14 FMAs),
//    which keeps the kernel at ~110 registers instead of 168-195 when the taps sat in registers;
//  * LayerNorm statistics are fp32; the R*7 per-pixel partial sums are reduce-scattered inside each 16-lane group
//    (30 shuffles for 28 pixels) and combined across the C/32 groups through shared memory in a FIXED order, so a
//    clip's result is bit-identical whatever else is in the batch.  The fp32 instantiation uses the two-pass
//    variance of F.layer_norm; the bf16 one a single pass (sum and sum of squares together).
// =============================================================================================
constexpr int DW_R = 4;

// Sum NV (= 32 or 64) per-thread values over the 16 lanes of a half-warp.  On return lane l (0..15) holds in
// v[0 .. NV/16) the totals of values [ (NV/16) * rev(l) ... ), where rev is given by slot_of_lane below.
template <int NV>
__device__ __forceinline__ void halfwarp_reduce_scatter(float (&v)[NV], int lane) {
#pragma unroll
  for (int off = 8, n = NV / 2; off >= 1; off >>= 1, n >>= 1) {
    const bool up = lane & off;
#pragma unroll
    for (int i = 0; i < n; ++i) {
      const float send = up ? v[i] : v[i + n];
      const float keep = up ? v[i + n] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
}
// first value index owned by `lane` after halfwarp_reduce_scatter<NV>: bit 3 selects the upper half, bit 2 the
// upper quarter, ...
template <int NV>
__device__ __forceinline__ int slot_of_lane(int lane) {
  return ((lane & 8) ? NV / 2 : 0) + ((lane & 4) ? NV / 4 : 0) + ((lane & 2) ? NV / 8 : 0) + ((lane & 1) ? NV / 16 : 0);
}

// resident blocks the register budget is capped for: 5 x 96, 2 x 192 or 1 x 384 threads (15 / 12 / 12 warps per SM)
constexpr int dw_min_blocks(int threads) { return threads <= 96 ? 5 : (threads <= 192 ? 2 : 1); }

// RAG: clip b has valid[b] rows (clamped to [0, H]); rows past it are read as the conv's zero padding and not written.
template <typename T, int C, int S, int PF, bool RAG = false>
__global__ void __launch_bounds__(S* C / 2, dw_min_blocks(S* C / 2))
    dwconv_ln_kernel(const T* __restrict__ x, const T* __restrict__ w, const float* __restrict__ bias,
                     const float* __restrict__ ln_w, const float* __restrict__ ln_b, T* __restrict__ y, int H,
                     int W, int groups_per_block, const int32_t* __restrict__ valid) {
  using P = Pair<T>;
  using PT = typename P::type;
  constexpr int R = DW_R;
  constexpr int NP = R * 7;         // 28 pixels per thread
  constexpr int TPS = C / 2;        // threads per strip
  constexpr int G = C / 32;         // half-warp groups per strip
  constexpr bool kTwoPass = sizeof(T) == 4;
  constexpr int NV = kTwoPass ? 32 : 64;   // values reduced per pass (28 sums [+ 28 sums of squares], padded)
  static_assert((S * TPS) % 32 == 0, "block must be whole warps (full-mask shuffles)");
  extern __shared__ __align__(16) float dsm[];
  float2* sw = reinterpret_cast<float2*>(dsm);                 // [49][TPS] taps as fp32 pairs
  float* part = dsm + 2 * 49 * TPS;                             // [S][G][NV]
  float* tot = part + S * G * NV;                               // [S][NV]
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int cp = tid % TPS;
  const int s = tid / TPS;
  const int grp = cp >> 4;
  const int w0 = (blockIdx.x * S + s) * 7;
  const int b = blockIdx.z;
  const PT* xp = reinterpret_cast<const PT*>(x) + (size_t)b * H * W * TPS + cp;
  PT* yp = reinterpret_cast<PT*>(y) + (size_t)b * H * W * TPS + cp;

  // Column halo: only the first / last strip of a row ever leaves the image, so two hoisted predicates replace
  // the 13 per-element bounds checks; rows outside the image are skipped as a whole (block-uniform).
  const bool left_ok = w0 > 0, right_ok = w0 + 7 < W;
  const PT* x0 = xp + ((ptrdiff_t)w0 - 3) * TPS;   // never dereferenced where the predicates are false
  auto load_row = [&](int ih, PT(&dst)[13]) {
    // A row outside the image is never USED (its FMA block is skipped below), so it needs no zero fill: its loads
    // are redirected to row 0 and issued unconditionally -- 7 of the 13 loads lose their predicate and the MOV that
    // zeroed the destination.  Only the 3 + 3 column-halo words are predicated (they do enter the FMAs).
    const bool row_ok = ih >= 0 && ih < H;
    const PT* row = x0 + (size_t)(row_ok ? ih : 0) * W * TPS;
#pragma unroll
    for (int j = 0; j < 13; ++j) {
      if (j < 3) dst[j] = left_ok ? __ldg(row + j * TPS) : PT{};
      else if (j >= 10) dst[j] = right_ok ? __ldg(row + j * TPS) : PT{};
      else dst[j] = __ldg(row + j * TPS);
    }
  };
  // The first PF input rows are requested BEFORE the tap fill so that their L2/HBM latency overlaps the fill's own
  // round trip and barrier (ncu: the serial prologue was ~30 % of a block's lifetime).
  static_assert((R + 6) % PF == 0, "prefetch ring must divide the row count");
  pdl_trigger();       // programmatic dependent launch (common.cuh); x is the previous kernel's output
  pdl_wait();
  const int Hv = RAG ? min(max(__ldg(valid + b), 0), H) : H;      // block-uniform
  PT nxt[PF][13];
#pragma unroll
  for (int k = 0; k < PF; ++k) load_row((int)blockIdx.y * groups_per_block * R - 3 + k, nxt[k]);

  // tap fill: 49 * C / 2 words per block.  Issued 7 loads at a time (the first version's one-load-per-iteration loop
  // cost ~12 serial L2 round trips per block, a third of a block's lifetime) and amortised over `groups_per_block`
  // row groups.
  {
    constexpr int PER_THREAD = (49 * TPS + S * TPS - 1) / (S * TPS);
    PT tmp[7];
#pragma unroll
    for (int i0 = 0; i0 < PER_THREAD; i0 += 7) {
#pragma unroll
      for (int u = 0; u < 7; ++u) {
        const int i = tid + (i0 + u) * S * TPS;
        tmp[u] = (i0 + u < PER_THREAD && i < 49 * TPS) ? __ldg(reinterpret_cast<const PT*>(w) + i) : PT{};
      }
#pragma unroll
      for (int u = 0; u < 7; ++u) {
        const int i = tid + (i0 + u) * S * TPS;
        if (i0 + u < PER_THREAD && i < 49 * TPS) sw[i] = P::unpack(tmp[u]);
      }
    }
  }
  const float2 bs = make_float2(bias[2 * cp], bias[2 * cp + 1]);
  const float2 gw = make_float2(ln_w[2 * cp], ln_w[2 * cp + 1]);
  const float2 gb = make_float2(ln_b[2 * cp], ln_b[2 * cp + 1]);
  __syncthreads();

  for (int grp_i = 0; grp_i < groups_per_block; ++grp_i) {
  const int h0 = (blockIdx.y * groups_per_block + grp_i) * R;
  if (h0 >= Hv) break;   // block-uniform

  float2 acc[R][7];
#pragma unroll
  for (int r = 0; r < R; ++r)
#pragma unroll
    for (int p = 0; p < 7; ++p) acc[r][p] = bs;

  const float2* swc = sw + cp;
#pragma unroll
  for (int i = 0; i < R + 6; ++i) {
    float2 in[13];
#pragma unroll
    for (int j = 0; j < 13; ++j) in[j] = P::unpack(nxt[i % PF][j]);
    // prefetch PF rows ahead; past the end of this group, the first rows of the block's next group
    if (i + PF < R + 6) load_row(h0 - 3 + i + PF, nxt[i % PF]);
    else if (grp_i + 1 < groups_per_block) load_row(h0 + R - 3 + (i + PF - (R + 6)), nxt[i % PF]);
    const int ih = h0 - 3 + i;
    if (ih >= 0 && ih < Hv) {                                   // zero padding contributes nothing (block-uniform)
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const int ky = i - r;                                   // compile-time after unrolling
        if (ky >= 0 && ky <= 6) {
#pragma unroll
          for (int kx = 0; kx < 7; ++kx) {
            const float2 wv = swc[(ky * 7 + kx) * TPS];
#pragma unroll
            for (int p = 0; p < 7; ++p) acc[r][p] = __ffma2_rn(in[p + kx], wv, acc[r][p]);   // packed fp32x2 FMA (sm_100)
          }
        }
      }
    }
  }

  // ---- LayerNorm over C -------------------------------------------------------------------------------
  float* my_part = part + (s * G + grp) * NV;
  float* my_tot = tot + s * NV;
  constexpr int PER_LANE = NV / 16;
  auto block_allreduce = [&](float(&v)[NV]) {
    halfwarp_reduce_scatter<NV>(v, lane);
    const int slot = slot_of_lane<NV>(lane & 15);
#pragma unroll
    for (int q = 0; q < PER_LANE; ++q) my_part[slot + q] = v[q];
    __syncthreads();
    for (int q = cp; q < NV; q += TPS) {                        // fixed-order sum over the G groups
      float t = part[(s * G) * NV + q];
#pragma unroll
      for (int g = 1; g < G; ++g) t += part[(s * G + g) * NV + q];
      my_tot[q] = t;
    }
    __syncthreads();
  };
  if (kTwoPass) {
    float mean[NP], rstd[NP];
    float v[NV];
#pragma unroll
    for (int q = 0; q < NV; ++q) v[q] = q < NP ? acc[q / 7][q % 7].x + acc[q / 7][q % 7].y : 0.f;
    block_allreduce(v);
#pragma unroll
    for (int q = 0; q < NP; ++q) {
      mean[q] = my_tot[q] * (1.0f / C);
      const float dx = acc[q / 7][q % 7].x - mean[q], dy = acc[q / 7][q % 7].y - mean[q];
      v[q] = dx * dx + dy * dy;
    }
#pragma unroll
    for (int q = NP; q < NV; ++q) v[q] = 0.f;
    block_allreduce(v);   // the first barrier inside also orders the my_tot reads above before its rewrite
#pragma unroll
    for (int q = 0; q < NP; ++q) rstd[q] = rsqrtf(my_tot[q] * (1.0f / C) + 1e-6f);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int h = h0 + r;
      if (h >= Hv) break;
      PT* orow = yp + ((size_t)h * W + w0) * TPS;
#pragma unroll
      for (int p = 0; p < 7; ++p) {
        const int q = r * 7 + p;
        const float sc = rstd[q];
        orow[(size_t)p * TPS] = P::pack((acc[r][p].x - mean[q]) * sc * gw.x + gb.x, (acc[r][p].y - mean[q]) * sc * gw.y + gb.y);
      }
    }
  } else {
    // one pass: sums and sums of squares reduced together; ONE thread per pixel turns them into (rstd, -mean*rstd)
    // so every other thread only does  out = acc * (rstd*g) + (-mean*rstd*g + b)  with three packed fp32x2 ops
    float v[NV];
#pragma unroll
    for (int q = 0; q < 32; ++q) {
      const float2 a2 = q < NP ? acc[q / 7][q % 7] : make_float2(0.f, 0.f);
      const float2 sq = __fmul2_rn(a2, a2);
      v[q] = a2.x + a2.y;
      v[32 + q] = sq.x + sq.y;
    }
    halfwarp_reduce_scatter<NV>(v, lane);
    const int slot = slot_of_lane<NV>(lane & 15);
#pragma unroll
    for (int q = 0; q < PER_LANE; ++q) my_part[slot + q] = v[q];
    __syncthreads();
    float2* my_stat = reinterpret_cast<float2*>(my_tot);       // [32] (rstd, -mean * rstd)
    if (cp < 32) {
      float su = part[(s * G) * NV + cp], sq = part[(s * G) * NV + 32 + cp];
#pragma unroll
      for (int g = 1; g < G; ++g) {                             // fixed order
        su += part[(s * G + g) * NV + cp];
        sq += part[(s * G + g) * NV + 32 + cp];
      }
      const float mean = su * (1.0f / C);
      const float var = fmaxf(sq * (1.0f / C) - mean * mean, 0.f);
      const float rs = rsqrtf(var + 1e-6f);
      my_stat[cp] = make_float2(rs, -mean * rs);
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int h = h0 + r;
      if (h >= Hv) break;
      PT* orow = yp + ((size_t)h * W + w0) * TPS;
#pragma unroll
      for (int p = 0; p < 7; ++p) {
        const float2 st = my_stat[r * 7 + p];
        const float2 sc = __fmul2_rn(make_float2(st.x, st.x), gw);
        const float2 of = __ffma2_rn(make_float2(st.y, st.y), gw, gb);
        const float2 o = __ffma2_rn(acc[r][p], sc, of);
        orow[(size_t)p * TPS] = P::pack(o.x, o.y);
      }
    }
  }
  }  // row groups of this block
}

// =============================================================================================
// channels_first LayerNorm + 2x2 patch gather (reference convnext.py:231-234).
// C/24 lanes per INPUT pixel, 24 channels (three 16-byte vectors in bf16) per lane: every load / store instruction
// of a warp moves 512 contiguous-per-pixel bytes, statistics are reduced with log2(C/24) shuffles, and each lane
// works on NPIX pixels at once so their loads overlap.  (First version: 4-byte loads, 28 % of HBM roofline.)
// =============================================================================================
// GP: x is group-planar [C/8][B*H*W][8] (bf16 only; the residual stream of the stages whose depthwise conv runs on the
// tensor cores); the patch matrix `a` is row-major either way.
template <typename T, int C, bool GP = false>
__global__ void __launch_bounds__(256, 3)
    ln_patchify_kernel(const T* __restrict__ x, const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                       T* __restrict__ a, int B, int H, int W) {
  constexpr int CH = 24;                      // channels per lane
  constexpr int LPP = C / CH;                 // lanes per pixel: 4 / 8 / 16
  constexpr int VE = 16 / (int)sizeof(T);     // elements per 16-byte vector
  constexpr int NV = CH / VE;                 // vectors per lane: 3 (bf16) / 6 (fp32)
  constexpr int NPIX = 2;                     // pixels in flight per lane group
  static_assert(C % CH == 0 && (LPP & (LPP - 1)) == 0 && LPP <= 32, "lane split");
  const int lig = threadIdx.x % LPP;          // lane in group
  const int Ho = H / 2, Wo = W / 2;
  const long long total = (long long)B * Ho * 2 * Wo * 2;
  const long long grp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / LPP;
  // the affine vectors are read (L1-resident) where they are used instead of living in 48 registers across the
  // loads: 3 blocks per SM instead of 2 keep more bytes in flight (ncu: 21 % occupancy, 42-59 % of HBM before)
  const float* gp = ln_w + lig * CH;
  const float* bp = ln_b + lig * CH;
  pdl_trigger();       // programmatic dependent launch (common.cuh); x is the previous kernel's output
  pdl_wait();
  float v[NPIX][CH];
  size_t dst_off[NPIX];
  bool ok[NPIX];
#pragma unroll
  for (int q = 0; q < NPIX; ++q) {
    const long long pix = grp * NPIX + q;
    ok[q] = pix < total;
    const long long pp = ok[q] ? pix : 0;
    const int wi = (int)(pp % (Wo * 2));
    const int hi = (int)((pp / (Wo * 2)) % (Ho * 2));
    const int b = (int)(pp / ((long long)Wo * 2 * Ho * 2));
    const size_t pix_in = ((size_t)b * H + hi) * W + wi;
    const size_t gp_stride = ((size_t)B * H * W + 127) / 128 * 128;     // plane stride in 16-byte vectors (rows padded to 128)
    const T* src = GP ? x + ((size_t)(lig * NV) * gp_stride + pix_in) * VE : x + pix_in * C + lig * CH;
    const size_t m = ((size_t)b * Ho + (hi >> 1)) * Wo + (wi >> 1);
    dst_off[q] = m * (size_t)(4 * C) + (size_t)((hi & 1) * 2 + (wi & 1)) * C + lig * CH;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const uint4 raw = __ldg(reinterpret_cast<const uint4*>(src) + (GP ? j * gp_stride : (size_t)j));
      if (sizeof(T) == 2) {
        float2 f;
        f = Pair<bf16>::unpack(raw.x); v[q][8 * j + 0] = f.x; v[q][8 * j + 1] = f.y;
        f = Pair<bf16>::unpack(raw.y); v[q][8 * j + 2] = f.x; v[q][8 * j + 3] = f.y;
        f = Pair<bf16>::unpack(raw.z); v[q][8 * j + 4] = f.x; v[q][8 * j + 5] = f.y;
        f = Pair<bf16>::unpack(raw.w); v[q][8 * j + 6] = f.x; v[q][8 * j + 7] = f.y;
      } else {
        v[q][4 * j + 0] = __uint_as_float(raw.x);
        v[q][4 * j + 1] = __uint_as_float(raw.y);
        v[q][4 * j + 2] = __uint_as_float(raw.z);
        v[q][4 * j + 3] = __uint_as_float(raw.w);
      }
    }
  }
#pragma unroll
  for (int q = 0; q < NPIX; ++q) {
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < CH; ++j) sum += v[q][j];
#pragma unroll
    for (int o = LPP / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float mean = sum / C;
    float sq = 0.f;
#pragma unroll
    for (int j = 0; j < CH; ++j) {
      v[q][j] -= mean;
      sq = fmaf(v[q][j], v[q][j], sq);
    }
#pragma unroll
    for (int o = LPP / 2; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    const float rstd = 1.0f / sqrtf(sq / C + 1e-6f);
    if (ok[q]) {
      T* dst = a + dst_off[q];
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        uint4 o4;
        if (sizeof(T) == 2) {
          const int k = 8 * j;
          const float4 g0 = __ldg(reinterpret_cast<const float4*>(gp + k)), g1 = __ldg(reinterpret_cast<const float4*>(gp + k + 4));
          const float4 b0 = __ldg(reinterpret_cast<const float4*>(bp + k)), b1 = __ldg(reinterpret_cast<const float4*>(bp + k + 4));
          o4.x = Pair<bf16>::pack(v[q][k + 0] * rstd * g0.x + b0.x, v[q][k + 1] * rstd * g0.y + b0.y);
          o4.y = Pair<bf16>::pack(v[q][k + 2] * rstd * g0.z + b0.z, v[q][k + 3] * rstd * g0.w + b0.w);
          o4.z = Pair<bf16>::pack(v[q][k + 4] * rstd * g1.x + b1.x, v[q][k + 5] * rstd * g1.y + b1.y);
          o4.w = Pair<bf16>::pack(v[q][k + 6] * rstd * g1.z + b1.z, v[q][k + 7] * rstd * g1.w + b1.w);
        } else {
          const int k = 4 * j;
          const float4 g0 = __ldg(reinterpret_cast<const float4*>(gp + k));
          const float4 b0 = __ldg(reinterpret_cast<const float4*>(bp + k));
          o4.x = __float_as_uint(v[q][k + 0] * rstd * g0.x + b0.x);
          o4.y = __float_as_uint(v[q][k + 1] * rstd * g0.y + b0.y);
          o4.z = __float_as_uint(v[q][k + 2] * rstd * g0.z + b0.z);
          o4.w = __float_as_uint(v[q][k + 3] * rstd * g0.w + b0.w);
        }
        reinterpret_cast<uint4*>(dst)[j] = o4;
      }
    }
  }
}

// =============================================================================================
// head (reference convnext.py:279-285, 321-325), two kernels:
//   pool:   grid (C/64, B): mean over mel (W), then max_t + mean_t  -> pooled (B, C) fp32
//   ln_fc:  grid (B, 8):    LayerNorm(C) (recomputed per block, 768 values) -> scene; 1/8 of the fc rows -> logits,
//           sigmoid -> probs
// =============================================================================================
// RAG: clip b pools over its first valid[b] rows (clamped to [1, H]).
template <typename T, bool RAG = false>
__global__ void __launch_bounds__(256)
    head_pool_kernel(const T* __restrict__ x, float* __restrict__ pooled, int H, int W, int C, const int32_t* __restrict__ valid) {
  using P = Pair<T>;
  using PT = typename P::type;
  __shared__ float2 smax[8][32], ssum[8][32];
  pdl_trigger();       // programmatic dependent launch (common.cuh)
  pdl_wait();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const int cp = blockIdx.x * 32 + lane;                 // channel pair
  const PT* xb = reinterpret_cast<const PT*>(x) + (size_t)b * H * W * (C / 2) + cp;
  const int Hv = RAG ? min(max(__ldg(valid + b), 1), H) : H;
  float2 mx = make_float2(-INFINITY, -INFINITY), sm = make_float2(0.f, 0.f);
  const float inv_w = 1.0f / W;
  for (int h = warp; h < Hv; h += 8) {
    float2 s = make_float2(0.f, 0.f);
    for (int wv = 0; wv < W; ++wv) {
      const float2 f = P::unpack(__ldg(xb + ((size_t)h * W + wv) * (C / 2)));
      s.x += f.x;
      s.y += f.y;
    }
    s.x *= inv_w;                                        // torch.mean(x, dim=3)   CX:279
    s.y *= inv_w;
    mx.x = fmaxf(mx.x, s.x);                             // torch.max(x, dim=2)    CX:280
    mx.y = fmaxf(mx.y, s.y);
    sm.x += s.x;                                         // torch.mean(x, dim=2)   CX:281
    sm.y += s.y;
  }
  smax[warp][lane] = mx;
  ssum[warp][lane] = sm;
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int i = 1; i < 8; ++i) {                        // fixed order
      mx.x = fmaxf(mx.x, smax[i][lane].x);
      mx.y = fmaxf(mx.y, smax[i][lane].y);
      sm.x += ssum[i][lane].x;
      sm.y += ssum[i][lane].y;
    }
    *reinterpret_cast<float2*>(pooled + (size_t)b * C + 2 * cp) = make_float2(mx.x + sm.x / Hv, mx.y + sm.y / Hv);  // CX:282
  }
}

__device__ __forceinline__ float block_sum_256(float v, float* scratch) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) t += scratch[i];
  return t;
}

__global__ void __launch_bounds__(256)
    head_ln_fc_kernel(const float* __restrict__ pooled, const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                      const float* __restrict__ fc_w, const float* __restrict__ fc_b, float* __restrict__ scene,
                      float* __restrict__ logits, float* __restrict__ probs, int C, int n_cls) {
  constexpr int MAXC = 4;  // C <= 1024
  extern __shared__ float sv[];  // C floats
  __shared__ float scratch[8];
  pdl_trigger();       // programmatic dependent launch (common.cuh); `pooled` is head_pool's output
  pdl_wait();
  const int b = blockIdx.x;
  const int tid = threadIdx.x;
  float val[MAXC], part = 0.f;
#pragma unroll
  for (int j = 0; j < MAXC; ++j) {
    const int c = tid + 256 * j;
    val[j] = (c < C) ? pooled[(size_t)b * C + c] : 0.f;
    part += val[j];
  }
  const float mean = block_sum_256(part, scratch) / C;
  part = 0.f;
#pragma unroll
  for (int j = 0; j < MAXC; ++j) {
    const int c = tid + 256 * j;
    if (c < C) {
      val[j] -= mean;
      part += val[j] * val[j];
    }
  }
  const float rstd = 1.0f / sqrtf(block_sum_256(part, scratch) / C + 1e-6f);  // nn.LayerNorm(768, eps 1e-6) CX:256
#pragma unroll
  for (int j = 0; j < MAXC; ++j) {
    const int c = tid + 256 * j;
    if (c < C) {
      const float o = val[j] * rstd * ln_w[c] + ln_b[c];
      sv[c] = o;
      if (blockIdx.y == 0) scene[(size_t)b * C + c] = o;
    }
  }
  __syncthreads();
  if (n_cls <= 0) return;
  const int lane = tid & 31, warp = tid >> 5;
  const int per = (n_cls + gridDim.y - 1) / gridDim.y;
  const int o_end = min(n_cls, (int)(blockIdx.y + 1) * per);
  for (int o = blockIdx.y * per + warp; o < o_end; o += 8) {
    const float* wr = fc_w + (size_t)o * C;
    float acc = 0.f;
    for (int k = lane * 4; k < C; k += 128) {
      const float4 w4 = __ldg(reinterpret_cast<const float4*>(wr + k));
      acc = fmaf(w4.x, sv[k], acc);
      acc = fmaf(w4.y, sv[k + 1], acc);
      acc = fmaf(w4.z, sv[k + 2], acc);
      acc = fmaf(w4.w, sv[k + 3], acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      const float lg = acc + fc_b[o];
      logits[(size_t)b * n_cls + o] = lg;
      probs[(size_t)b * n_cls + o] = 1.0f / (1.0f + expf(-lg));
    }
  }
}

// =============================================================================================
// NHWC (act dtype) -> NCHW fp32
// =============================================================================================
// RAG: rows of clip b at or past valid[b] (clamped to [0, H]) are written as zeros and not read.
template <typename T, bool RAG = false>
__global__ void nhwc_to_nchw_kernel(const T* __restrict__ x, float* __restrict__ out, int HW, int C, int W,
                                    const int32_t* __restrict__ valid) {
  __shared__ float tile[32][33];
  pdl_trigger();       // programmatic dependent launch (common.cuh)
  pdl_wait();
  const int b = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const T* xb = x + (size_t)b * HW * C;
  float* ob = out + (size_t)b * HW * C;
  const int pv = RAG ? min(max(__ldg(valid + b), 0), HW / W) * W : HW;      // valid pixels of this clip
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int p = p0 + i, c = c0 + threadIdx.x;
    if (p < HW && c < C) tile[i][threadIdx.x] = p < pv ? to_float(xb[(size_t)p * C + c]) : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, p = p0 + threadIdx.x;
    if (p < HW && c < C) ob[(size_t)c * HW + p] = tile[threadIdx.x][i];
  }
}

// =============================================================================================
// polyphase sinc resampler + pad / crop (reference demo_convnext.py:52-67 via torchaudio.functional.resample).
// Thread per output sample; a warp's lanes share the input window (broadcast loads) and read consecutive phases of
// the transposed tap table (coalesced).  One clip per demo call: ~150 MFLOP, latency-bound, not a hot kernel.
// =============================================================================================
__global__ void __launch_bounds__(256)
    resample_fit_kernel(const float* __restrict__ x, int ld_in, const float* __restrict__ taps, float* __restrict__ out,
                        int ld_out, int L_in, int orig, int newf, int width, int n_out, long long target) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_out) return;
  const float* xb = x + (size_t)blockIdx.y * ld_in;
  float acc = 0.f;
  if (i < target) {
    const int f = i / newf, p = i - f * newf;
    const long long base = (long long)f * orig - width;
    const int K = 2 * width + orig;
    for (int k = 0; k < K; ++k) {
      const long long idx = base + k;
      const float v = (idx >= 0 && idx < L_in) ? __ldg(xb + idx) : 0.f;
      acc = fmaf(__ldg(taps + (size_t)k * newf + p), v, acc);
    }
  }
  out[(size_t)blockIdx.y * ld_out + i] = acc;
}

// ---- segmented resampler: many recordings of any length packed in one buffer, 64-bit indices ----------------------
// Segment s is (in_off, in_len, out_off, out_len) int64: output j of the segment is what resample_fit_kernel computes for
// a row of in_len samples (frame f = j / newf, phase p = j % newf, the same fmaf chain over k = 0..K-1), with the input
// zero outside [0, in_len) of the SEGMENT.  Each entry is clamped to x_len / out_len, so no table value can make the
// kernel read or write outside its buffers.
//
// A block computes one tile: RS_THREADS / 32 warps, lanes = 32 consecutive frames, each thread RS_R consecutive phases
// (one float4 of taps per k, reused by its RS_R outputs; every output keeps its own sequential k order).  The tile's
// P phases' taps (K x P) and its input span ((F-1) * orig + K samples, converted to fp32 and zero-filled outside the
// segment) are staged in shared memory once, so the tap table is read from global memory once per block instead of
// once per output.  Tiles of all segments form one 1-D grid: tile_start[s] is segment s's first tile (a host-built
// prefix over ceil(frames / F) * G tiles per segment), which the block finds by binary search.  So one launch spreads
// a single long segment over every SM and also serves thousands of short clips.
constexpr int RS_R = 4, RS_WARPS = 8, RS_THREADS = 32 * RS_WARPS;
constexpr int RS_MAX_SMEM = 227 * 1024;

struct ResampleTiling {
  int P, F, G;          // phases and frames per tile, phase groups per frame tile
  long long smem;       // dynamic shared memory bytes
};

// Phase warps WP = the smallest power of two >= ceil(newf / RS_R), at most RS_WARPS; the other warps take more frames.
static inline ResampleTiling resample_tiling(int orig, int newf, int width) {
  const int quads = (newf + RS_R - 1) / RS_R;
  int wp = 1;
  while (wp < quads && wp < RS_WARPS) wp *= 2;
  ResampleTiling t;
  t.P = wp * RS_R;
  t.F = 32 * (RS_WARPS / wp);
  t.G = (newf + t.P - 1) / t.P;
  const long long K = 2LL * width + orig;
  t.smem = (K * t.P + (long long)(t.F - 1) * orig + K) * (long long)sizeof(float);
  return t;
}

//
// STREAM (acx_resample_stream): segment s is a live stream whose input and output are rings.  Its row is 8 int64:
// (in_base, in_cap, in_end, f0, n_out, out_base, out_cap, out_mirror).  Input sample idx of the stream is read from
// x[in_base + idx mod in_cap] and is zero for idx < 0 or idx >= in_end.  The block computes outputs f0 * newf + jl for
// jl < n_out (f0 a 64-bit stream frame), each by the same fmaf chain as above, and writes output j to
// out[out_base + j mod out_cap], and also to out[out_base + out_cap + j mod out_cap] when j mod out_cap < out_mirror.
template <typename TIn, bool STREAM = false>
__global__ void __launch_bounds__(RS_THREADS)
    resample_segments_kernel(const TIn* __restrict__ x, long long x_len, const long long* __restrict__ seg,
                             const long long* __restrict__ tile_start, int S, const float* __restrict__ taps, int orig,
                             int newf, int width, int P, int F, int G, float* __restrict__ out, long long out_len) {
  extern __shared__ float4 rs_smem[];
  const int K = 2 * width + orig;
  float* s_taps = reinterpret_cast<float*>(rs_smem);      // [K][P]
  float* s_x = s_taps + (size_t)K * P;                     // [(F-1) * orig + K]
  const long long tile = blockIdx.x;
  int lo = 0, hi = S - 1;                                  // last segment whose first tile is <= this one
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(tile_start + mid) <= tile) lo = mid; else hi = mid - 1;
  }
  const long long local = tile - __ldg(tile_start + lo);
  if (local < 0) return;
  const long long* e = seg + (STREAM ? 8 : 4) * (size_t)lo;
  long long in_off, in_len, out_off, n_out, in_cap = 0, fbase = 0, out_cap = 0, out_mirror = 0;
  if constexpr (STREAM) {
    in_off = min(max(__ldg(e), 0LL), x_len);
    in_cap = min(max(__ldg(e + 1), 0LL), x_len - in_off);
    in_len = max(__ldg(e + 2), 0LL);                       // in_end: samples of the stream received so far
    // bounded so that every stream index below ((fbase + tile frames) * orig, fbase * newf + j) fits in int64
    fbase = min(max(__ldg(e + 3), 0LL), (1LL << 62) / max(orig, newf));
    n_out = max(__ldg(e + 4), 0LL);
    out_off = min(max(__ldg(e + 5), 0LL), out_len);
    out_cap = min(max(__ldg(e + 6), 0LL), out_len - out_off);
    out_mirror = min(max(__ldg(e + 7), 0LL), min(out_cap, out_len - out_off - out_cap));
    if (in_cap < 1 || out_cap < 1) return;
  } else {
    in_off = min(max(__ldg(e), 0LL), x_len);
    in_len = min(max(__ldg(e + 1), 0LL), x_len - in_off);
    out_off = min(max(__ldg(e + 2), 0LL), out_len);
    n_out = min(max(__ldg(e + 3), 0LL), out_len - out_off);
  }
  const long long ft = local / G;
  const int p0 = (int)(local - ft * G) * P;
  const long long f0 = ft * F;
  if (f0 * newf >= n_out) return;                          // whole block: no barrier is skipped by part of it

  for (int i = threadIdx.x; i < K * P; i += RS_THREADS) {
    const int k = i / P, p = p0 + (i - k * P);
    s_taps[i] = p < newf ? __ldg(taps + (size_t)k * newf + p) : 0.f;
  }
  const TIn* xs = x + in_off;
  const long long i0 = (fbase + f0) * orig - width;
  const int span = (F - 1) * orig + K;
  if constexpr (STREAM) {
    long long slot = i0 % in_cap;                          // the span's first ring slot, reduced once
    if (slot < 0) slot += in_cap;
    slot += threadIdx.x;
    while (slot >= in_cap) slot -= in_cap;
    for (int i = threadIdx.x; i < span; i += RS_THREADS) {
      const long long idx = i0 + i;
      s_x[i] = (idx >= 0 && idx < in_len) ? load_sample(xs + slot) : 0.f;
      slot += RS_THREADS;
      while (slot >= in_cap) slot -= in_cap;               // once when in_cap >= RS_THREADS
    }
  } else {
    for (int i = threadIdx.x; i < span; i += RS_THREADS) {
      const long long idx = i0 + i;
      s_x[i] = (idx >= 0 && idx < in_len) ? load_sample(xs + idx) : 0.f;
    }
  }
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wp = P / RS_R;
  const int pl = (warp % wp) * RS_R;                       // first of this thread's RS_R phases in the tile
  const int fl = (warp / wp) * 32 + lane;                  // this thread's frame in the tile
  const float* xv = s_x + fl * orig;
  const float4* tv = reinterpret_cast<const float4*>(s_taps + pl);
  const int tstride = P / RS_R;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 4
  for (int k = 0; k < K; ++k) {
    const float v = xv[k];
    const float4 t = tv[k * tstride];
    a0 = fmaf(t.x, v, a0);
    a1 = fmaf(t.y, v, a1);
    a2 = fmaf(t.z, v, a2);
    a3 = fmaf(t.w, v, a3);
  }
  const int p = p0 + pl;
  const long long j = (f0 + fl) * newf + p;
  float* o = out + out_off;
  if constexpr (STREAM) {
    const float a[RS_R] = {a0, a1, a2, a3};
    long long slot = (fbase * newf + j) % out_cap;        // ring slot of stream output fbase * newf + j
#pragma unroll
    for (int r = 0; r < RS_R; ++r) {
      if (p + r < newf && j + r < n_out) {
        o[slot] = a[r];
        if (slot < out_mirror) o[out_cap + slot] = a[r];
      }
      if (++slot == out_cap) slot = 0;
    }
  } else {
    if (p < newf && j < n_out) o[j] = a0;
    if (p + 1 < newf && j + 1 < n_out) o[j + 1] = a1;
    if (p + 2 < newf && j + 2 < n_out) o[j + 2] = a2;
    if (p + 3 < newf && j + 3 < n_out) o[j + 3] = a3;
  }
}

// ---- live streams: one push's chunks scattered into every stream's ring in one launch -------------------------------
// tab is a DEVICE (S, 6) int64 table, row s = (src_off, n, ring_base, cap, pos, mirror): chunk s is src[src_off, src_off
// + n), and its sample i goes to ring[ring_base + (pos + i) mod cap], and also to ring[ring_base + cap + (pos + i) mod cap]
// when that slot is below `mirror`.  Rows are in src order (src_off non-decreasing); a thread finds its sample's row by
// binary search, so one launch serves one long chunk or thousands of short ones.  n <= cap, mirror <= cap and the region
// [ring_base, ring_base + cap + mirror) inside ring_len are enforced by clamping: no table value writes outside its row's
// region of the ring.  int16 PCM is converted x / 32767 with a correctly rounded division (load_sample).
template <typename TIn>
__global__ void __launch_bounds__(256)
    stream_append_kernel(const TIn* __restrict__ src, long long src_len, const long long* __restrict__ tab, int S,
                         float* __restrict__ ring, long long ring_len) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= src_len) return;
  int lo = 0, hi = S - 1;                                  // last row whose chunk starts at or before g
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(tab + 6 * (size_t)mid) <= g) lo = mid; else hi = mid - 1;
  }
  const long long* e = tab + 6 * (size_t)lo;
  const long long base = min(max(__ldg(e + 2), 0LL), ring_len);
  const long long cap = min(max(__ldg(e + 3), 0LL), ring_len - base);
  const long long n = min(max(__ldg(e + 1), 0LL), cap);
  const long long i = g - min(max(__ldg(e), 0LL), src_len);
  if (i < 0 || i >= n) return;
  const long long mirror = min(max(__ldg(e + 5), 0LL), min(cap, ring_len - base - cap));
  long long pos = max(__ldg(e + 4), 0LL);
  if (pos >= cap) pos %= cap;                              // the planner passes pos < cap; any other value is reduced
  long long slot = pos + i;                                // < 2 cap: no overflow for any table value
  if (slot >= cap) slot -= cap;
  const float v = load_sample(src + g);
  ring[base + slot] = v;
  if (slot < mirror) ring[base + cap + slot] = v;
}

// ---- launch helpers ---------------------------------------------------------------------------
template <typename T, int C, int S, int PF = 2, bool RAG = false>
static int launch_dwconv(const void* x, const void* w, const float* bias, const float* ln_w, const float* ln_b,
                         void* y, int B, int H, int W, const int32_t* valid, cudaStream_t st) {
  const int strips = W / 7;
  ACX_CHECK(strips % S == 0, ACX_ERR_ARG, "dwconv_ln: W/7=%d not a multiple of strips-per-block %d", strips, S);
  constexpr int NV = sizeof(T) == 4 ? 32 : 64;
  constexpr int SMEM = (2 * 49 * (C / 2) + S * (C / 32) * NV + S * NV) * (int)sizeof(float);
  auto kern = dwconv_ln_kernel<T, C, S, PF, RAG>;
  ACX_SET_MAX_SMEM(kern, SMEM);
  const int row_groups = ceil_div(H, DW_R);
  // Row groups per block.  With the first input rows requested ahead of the tap fill (and the next group's rows
  // ahead of the LayerNorm phase) one group per block is fastest everywhere except the tiny stage-4 maps, where the
  // 150 KB tap fill dominates (measured, 64 clips: C=768 0.137 / 0.133 / 0.129 ms at 1 / 2 / 4 groups; C=384
  // 0.688 / 0.703 / 0.779; C=96 0.783 / 0.807 / 0.829).  ACX_DW_GPB overrides for experiments.
  static const int gpb_env = [] { const char* e = getenv("ACX_DW_GPB"); return e ? atoi(e) : 0; }();
  int gpb = (C >= 768 && row_groups >= 4) ? 4 : 1;
  if (gpb_env > 0) gpb = gpb_env < row_groups ? gpb_env : row_groups;
  dim3 grid(strips / S, ceil_div(row_groups, gpb), B);
  ACX_CUDA(launch_pdl(kern, grid, dim3(S * C / 2), SMEM, st, 1, PDL_SMALL, reinterpret_cast<const T*>(x), reinterpret_cast<const T*>(w), bias,
                      ln_w, ln_b, reinterpret_cast<T*>(y), H, W, gpb, valid));
  return ACX_OK;
}

template <typename T, bool RAG>
static int dispatch_dwconv(const void* x, const void* w, const float* bias, const float* ln_w, const float* ln_b,
                           void* y, int B, int H, int W, int C, const int32_t* valid, cudaStream_t st) {
  const int strips = W / 7;
  // A/B switches (development only): ACX_DW_PF=1 -> one-row prefetch, ACX_DW_NARROW=1 -> half-width blocks
  static const bool pf1 = [] { const char* e = getenv("ACX_DW_PF"); return e && e[0] == '1'; }();
  static const bool narrow = [] { const char* e = getenv("ACX_DW_NARROW"); return e && e[0] == '1'; }();
#define ACX_DW_LAUNCH(CC, SS) \
  (pf1 ? launch_dwconv<T, CC, SS, 1, RAG>(x, w, bias, ln_w, ln_b, y, B, H, W, valid, st) \
       : launch_dwconv<T, CC, SS, 2, RAG>(x, w, bias, ln_w, ln_b, y, B, H, W, valid, st))
  switch (C) {
    case 96:
      if (strips % 4 == 0 && !narrow) return ACX_DW_LAUNCH(96, 4);
      if (strips % 2 == 0) return ACX_DW_LAUNCH(96, 2);
      set_error("dwconv_ln: C=96 needs an even number of 7-pixel strips per row (W=%d)", W);
      return ACX_ERR_UNSUPPORTED;
    case 192:
      if (strips % 2 == 0 && !narrow) return ACX_DW_LAUNCH(192, 2);
      return ACX_DW_LAUNCH(192, 1);
    case 384:
      return ACX_DW_LAUNCH(384, 1);
    case 768:
      return ACX_DW_LAUNCH(768, 1);
    default:
      set_error("dwconv_ln: unsupported channel count %d (ConvNeXt-Tiny dims are 96/192/384/768)", C);
      return ACX_ERR_UNSUPPORTED;
  }
#undef ACX_DW_LAUNCH
}

}  // namespace acx

namespace acx {
int launch_stem_umma(const float* logmel, const float* w, const float* bias, const float* ln_w, const float* ln_b,
                     void* out, int B, int T, int n_mels, int gp, const int32_t* valid, cudaStream_t st);   // stem_umma.cu
}
using namespace acx;

template <typename TIn>
static int wave_prep_launch(const TIn* wave, void* hi, void* lo, int B, int L, int n_fft, int ld_pad, int act_dtype,
                            int ld_wave, const int32_t* valid, void* stream, const long long* offsets = nullptr,
                            long long rec_len = 0) {
  ACX_CHECK(wave && hi && B > 0 && L > 0, ACX_ERR_ARG, "wave_prep: null pointer or empty batch");
  ACX_CHECK(ld_wave >= L, ACX_ERR_ARG, "wave_prep: row pitch %d < L=%d", ld_wave, L);
  ACX_CHECK(L > n_fft / 2, ACX_ERR_ARG, "wave_prep: reflect padding needs L > n_fft/2 (L=%d)", L);
  ACX_CHECK(ld_pad >= L + n_fft && ld_pad % 8 == 0, ACX_ERR_ARG, "wave_prep: ld_pad=%d must be >= L+n_fft and %%8==0",
            ld_pad);
  ACX_CHECK(B <= 65535, ACX_ERR_ARG, "wave_prep: batch %d exceeds gridDim.y", B);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  dim3 grid(ceil_div(ld_pad, 1024), B);
  ACX_CHECK(act_dtype != ACX_BF16 || lo != nullptr, ACX_ERR_ARG, "wave_prep: lo buffer required for bf16 split");
  constexpr bool kRagged = std::is_same<TIn, float>::value;     // ragged batches are fp32 waveforms only
  const int pad = n_fft / 2;
  if (offsets && valid && act_dtype == ACX_BF16)                // windows of one recording (fp32 or int16)
    wave_prep_kernel<true, TIn, true, true><<<grid, 256, 0, st>>>(wave, hi, lo, L, pad, ld_pad, L, valid, offsets, rec_len);
  else if (offsets && valid)
    wave_prep_kernel<false, TIn, true, true><<<grid, 256, 0, st>>>(wave, hi, lo, L, pad, ld_pad, L, valid, offsets, rec_len);
  else if (offsets && act_dtype == ACX_BF16)
    wave_prep_kernel<true, TIn, false, true><<<grid, 256, 0, st>>>(wave, hi, lo, L, pad, ld_pad, L, nullptr, offsets, rec_len);
  else if (offsets)
    wave_prep_kernel<false, TIn, false, true><<<grid, 256, 0, st>>>(wave, hi, lo, L, pad, ld_pad, L, nullptr, offsets, rec_len);
  else if (kRagged && valid && act_dtype == ACX_BF16)
    wave_prep_kernel<true, TIn, kRagged><<<grid, 256, 0, st>>>(wave, hi, lo, L, n_fft / 2, ld_pad, ld_wave, valid);
  else if (kRagged && valid)
    wave_prep_kernel<false, TIn, kRagged><<<grid, 256, 0, st>>>(wave, hi, lo, L, n_fft / 2, ld_pad, ld_wave, valid);
  else if (act_dtype == ACX_BF16)
    wave_prep_kernel<true, TIn><<<grid, 256, 0, st>>>(wave, hi, lo, L, n_fft / 2, ld_pad, ld_wave, nullptr);
  else
    wave_prep_kernel<false, TIn><<<grid, 256, 0, st>>>(wave, hi, lo, L, n_fft / 2, ld_pad, ld_wave, nullptr);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

template <typename TIn>
static int wave_prep_windows(const TIn* rec, long long rec_len, const long long* offsets, const int32_t* valid, void* hi,
                             void* lo, int B, int L, int n_fft, int ld_pad, int act_dtype, void* stream) {
  ACX_CHECK(rec && offsets, ACX_ERR_ARG, "wave_prep_windows: null recording or offsets");
  ACX_CHECK(rec_len >= n_fft / 2 + 1, ACX_ERR_ARG, "wave_prep_windows: rec_len=%lld must be > n_fft/2 (reflect padding)",
            rec_len);
  ACX_CHECK(B >= 1, ACX_ERR_ARG, "wave_prep_windows: empty batch B=%d", B);
  return wave_prep_launch<TIn>(rec, hi, lo, B, L, n_fft, ld_pad, act_dtype, L, valid, stream, offsets, rec_len);
}

extern "C" {

int acx_wave_prep(const float* wave, void* hi, void* lo, int B, int L, int n_fft, int ld_pad, int act_dtype,
                  void* stream) {
  return wave_prep_launch<float>(wave, hi, lo, B, L, n_fft, ld_pad, act_dtype, L, nullptr, stream);
}

int acx_wave_prep_ragged(const float* wave, void* hi, void* lo, int B, int L, int n_fft, int ld_pad, int act_dtype,
                         int ld_wave, const int32_t* valid, void* stream) {
  ACX_CHECK(valid, ACX_ERR_ARG, "wave_prep_ragged: null valid-length array");
  return wave_prep_launch<float>(wave, hi, lo, B, L, n_fft, ld_pad, act_dtype, ld_wave, valid, stream);
}

int acx_wave_prep_pcm16(const int16_t* pcm, void* hi, void* lo, int B, int L, int n_fft, int ld_pad, int act_dtype,
                        void* stream) {
  return wave_prep_launch<int16_t>(pcm, hi, lo, B, L, n_fft, ld_pad, act_dtype, L, nullptr, stream);
}

int acx_wave_prep_windows(const float* rec, long long rec_len, const long long* offsets, const int32_t* valid, void* hi,
                          void* lo, int B, int L, int n_fft, int ld_pad, int act_dtype, void* stream) {
  return wave_prep_windows<float>(rec, rec_len, offsets, valid, hi, lo, B, L, n_fft, ld_pad, act_dtype, stream);
}

int acx_wave_prep_pcm16_windows(const int16_t* rec, long long rec_len, const long long* offsets, const int32_t* valid,
                                void* hi, void* lo, int B, int L, int n_fft, int ld_pad, int act_dtype, void* stream) {
  return wave_prep_windows<int16_t>(rec, rec_len, offsets, valid, hi, lo, B, L, n_fft, ld_pad, act_dtype, stream);
}

int acx_power_mel_log(const float* spec, int ld_spec, int n_bins, const float* melT, const int32_t* mel_lo,
                      const int32_t* mel_hi, const float* bn_scale, const float* bn_shift, float* out, int rows,
                      int n_mels, void* stream) {
  ACX_CHECK(spec && melT && mel_lo && mel_hi && bn_scale && bn_shift && out, ACX_ERR_ARG, "power_mel_log: null pointer");
  ACX_CHECK(rows > 0 && n_bins > 0 && n_bins <= 8192, ACX_ERR_ARG, "power_mel_log: bad sizes");
  power_mel_log_kernel<<<rows, 256, n_bins * sizeof(float), reinterpret_cast<cudaStream_t>(stream)>>>(
      spec, ld_spec, n_bins, melT, mel_lo, mel_hi, bn_scale, bn_shift, out, rows, n_mels);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

static int stem_impl(const float* logmel, const float* w, const float* bias, const float* ln_w, const float* ln_b, void* out,
                     int B, int T, int n_mels, int act_dtype, const int32_t* valid, void* stream) {
  ACX_CHECK(logmel && w && bias && ln_w && ln_b && out, ACX_ERR_ARG, "stem: null pointer");
  ACX_CHECK(n_mels % 4 == 0 && B > 0 && T > 0, ACX_ERR_ARG, "stem: n_mels must be a multiple of 4");
  const int H0 = (T + 4) / 4 + 1, W0 = n_mels / 4;
  const long long total = (long long)B * H0 * W0;
  const int blocks = (int)((total + 127) / 128);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // bf16 mode: tensor-core stem (stem_umma.cu); ACX_STEM=simt selects the CUDA-core kernel for A/B timing
  static const bool stem_simt = [] { const char* e = getenv("ACX_STEM"); return e && e[0] == 's'; }();
  if (act_dtype == ACX_BF16 && !stem_simt)
    return launch_stem_umma(logmel, w, bias, ln_w, ln_b, out, B, T, n_mels, 0, valid, st);
  if (act_dtype == ACX_BF16) {
    const int smem = 19 * 96 * 4 + 4 * 32 * (96 * 2 + 16);
    auto kern = valid ? stem_kernel<bf16, true> : stem_kernel<bf16>;
    kern<<<blocks, 128, smem, st>>>(logmel, w, bias, ln_w, ln_b, reinterpret_cast<bf16*>(out), B, T, n_mels, H0, W0, valid);
  } else {
    const int smem = 19 * 96 * 4 + 4 * 32 * (96 * 4 + 16);
    auto kern = valid ? stem_kernel<float, true> : stem_kernel<float>;
    if (valid) ACX_SET_MAX_SMEM((stem_kernel<float, true>), smem);
    else ACX_SET_MAX_SMEM(stem_kernel<float>, smem);
    kern<<<blocks, 128, smem, st>>>(logmel, w, bias, ln_w, ln_b, reinterpret_cast<float*>(out), B, T, n_mels, H0, W0, valid);
  }
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

int acx_stem(const float* logmel, const float* w, const float* bias, const float* ln_w, const float* ln_b, void* out,
             int B, int T, int n_mels, int act_dtype, void* stream) {
  return stem_impl(logmel, w, bias, ln_w, ln_b, out, B, T, n_mels, act_dtype, nullptr, stream);
}

int acx_stem_ragged(const float* logmel, const float* w, const float* bias, const float* ln_w, const float* ln_b, void* out,
                    int B, int T, int n_mels, int act_dtype, const int32_t* valid, void* stream) {
  ACX_CHECK(valid, ACX_ERR_ARG, "stem_ragged: null valid-length array");
  return stem_impl(logmel, w, bias, ln_w, ln_b, out, B, T, n_mels, act_dtype, valid, stream);
}

static int dwconv_ln_impl(const void* x, const void* w, const float* bias, const float* ln_w, const float* ln_b, void* y,
                          int B, int H, int W, int C, int act_dtype, const int32_t* valid, void* stream) {
  ACX_CHECK(x && w && bias && ln_w && ln_b && y, ACX_ERR_ARG, "dwconv_ln: null pointer");
  ACX_CHECK(B > 0 && H > 0 && W > 0 && W % 7 == 0, ACX_ERR_ARG, "dwconv_ln: W=%d must be a positive multiple of 7", W);
  ACX_CHECK(B <= 65535, ACX_ERR_ARG, "dwconv_ln: batch %d exceeds gridDim.z", B);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (valid)
    return act_dtype == ACX_BF16 ? dispatch_dwconv<bf16, true>(x, w, bias, ln_w, ln_b, y, B, H, W, C, valid, st)
                                 : dispatch_dwconv<float, true>(x, w, bias, ln_w, ln_b, y, B, H, W, C, valid, st);
  return act_dtype == ACX_BF16 ? dispatch_dwconv<bf16, false>(x, w, bias, ln_w, ln_b, y, B, H, W, C, nullptr, st)
                               : dispatch_dwconv<float, false>(x, w, bias, ln_w, ln_b, y, B, H, W, C, nullptr, st);
}

int acx_dwconv_ln(const void* x, const void* w, const float* bias, const float* ln_w, const float* ln_b, void* y, int B,
                  int H, int W, int C, int act_dtype, void* stream) {
  return dwconv_ln_impl(x, w, bias, ln_w, ln_b, y, B, H, W, C, act_dtype, nullptr, stream);
}

int acx_dwconv_ln_ragged(const void* x, const void* w, const float* bias, const float* ln_w, const float* ln_b, void* y,
                         int B, int H, int W, int C, int act_dtype, const int32_t* valid, void* stream) {
  ACX_CHECK(valid, ACX_ERR_ARG, "dwconv_ln_ragged: null valid-length array");
  return dwconv_ln_impl(x, w, bias, ln_w, ln_b, y, B, H, W, C, act_dtype, valid, stream);
}

// bf16 tensor-core stem writing the group-planar layout [12][Mp][8] directly (Mp = B * H0 * 56 rounded up to 128)
int acx_stem_gp(const float* logmel, const float* w, const float* bias, const float* ln_w, const float* ln_b, void* out,
                int B, int T, int n_mels, void* stream) {
  ACX_CHECK(logmel && w && bias && ln_w && ln_b && out, ACX_ERR_ARG, "stem_gp: null pointer");
  ACX_CHECK(n_mels % 4 == 0 && B > 0 && T > 0, ACX_ERR_ARG, "stem_gp: n_mels must be a multiple of 4");
  return launch_stem_umma(logmel, w, bias, ln_w, ln_b, out, B, T, n_mels, 1, nullptr, reinterpret_cast<cudaStream_t>(stream));
}

int acx_stem_gp_ragged(const float* logmel, const float* w, const float* bias, const float* ln_w, const float* ln_b, void* out,
                       int B, int T, int n_mels, const int32_t* valid, void* stream) {
  ACX_CHECK(valid, ACX_ERR_ARG, "stem_gp_ragged: null valid-length array");
  ACX_CHECK(logmel && w && bias && ln_w && ln_b && out, ACX_ERR_ARG, "stem_gp: null pointer");
  ACX_CHECK(n_mels % 4 == 0 && B > 0 && T > 0, ACX_ERR_ARG, "stem_gp: n_mels must be a multiple of 4");
  return launch_stem_umma(logmel, w, bias, ln_w, ln_b, out, B, T, n_mels, 1, valid, reinterpret_cast<cudaStream_t>(stream));
}

int acx_ln_patchify(const void* x, const float* ln_w, const float* ln_b, void* a, int B, int H, int W, int C,
                    int act_dtype, void* stream) {
  ACX_CHECK(x && ln_w && ln_b && a, ACX_ERR_ARG, "ln_patchify: null pointer");
  ACX_CHECK((C == 96 || C == 192 || C == 384) && H >= 2 && W >= 2, ACX_ERR_ARG,
            "ln_patchify: unsupported shape C=%d H=%d W=%d (C must be 96, 192 or 384)", C, H, W);
  const long long total = (long long)B * (H / 2) * 2 * (W / 2) * 2;
  const long long lanes = (total + 1) / 2 * (C / 24);        // C/24 lanes per pixel, 2 pixels per lane group
  const int blocks = (int)((lanes + 255) / 256);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
#define ACX_LNP(TT, CC)                                                                                     \
  ACX_CUDA(launch_pdl(ln_patchify_kernel<TT, CC>, dim3(blocks), dim3(256), 0, st, 1, PDL_SMALL, reinterpret_cast<const TT*>(x), ln_w, \
                      ln_b, reinterpret_cast<TT*>(a), B, H, W))
  if (act_dtype == ACX_BF16) {
    if (C == 96) ACX_LNP(bf16, 96); else if (C == 192) ACX_LNP(bf16, 192); else ACX_LNP(bf16, 384);
  } else {
    if (C == 96) ACX_LNP(float, 96); else if (C == 192) ACX_LNP(float, 192); else ACX_LNP(float, 384);
  }
#undef ACX_LNP
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

// Same with a group-planar input x = [C/8][B*H*W][8] bf16 (stages 0 / 1 behind the tensor-core depthwise conv).
int acx_ln_patchify_gp(const void* x, const float* ln_w, const float* ln_b, void* a, int B, int H, int W, int C,
                       void* stream) {
  ACX_CHECK(x && ln_w && ln_b && a, ACX_ERR_ARG, "ln_patchify_gp: null pointer");
  ACX_CHECK((C == 96 || C == 192 || C == 384) && H >= 2 && W >= 2, ACX_ERR_ARG,
            "ln_patchify_gp: unsupported shape C=%d H=%d W=%d (C must be 96, 192 or 384)", C, H, W);
  const long long total = (long long)B * (H / 2) * 2 * (W / 2) * 2;
  const long long lanes = (total + 1) / 2 * (C / 24);
  const int blocks = (int)((lanes + 255) / 256);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  auto kern = C == 96 ? ln_patchify_kernel<bf16, 96, true> : C == 192 ? ln_patchify_kernel<bf16, 192, true> : ln_patchify_kernel<bf16, 384, true>;
  ACX_CUDA(launch_pdl(kern, dim3(blocks), dim3(256), 0, st, 1, PDL_SMALL, reinterpret_cast<const bf16*>(x), ln_w, ln_b, reinterpret_cast<bf16*>(a), B,
                      H, W));
  return ACX_OK;
}

static int head_impl(const void* x, const float* ln_w, const float* ln_b, const float* fc_w, const float* fc_b, float* pooled,
                     float* scene, float* logits, float* probs, int B, int H, int W, int C, int n_cls, int act_dtype,
                     const int32_t* valid, void* stream) {
  ACX_CHECK(x && ln_w && ln_b && scene && pooled, ACX_ERR_ARG, "head: null pointer");
  ACX_CHECK(n_cls == 0 || (fc_w && fc_b && logits && probs), ACX_ERR_ARG, "head: fc pointers required when n_cls>0");
  ACX_CHECK(C % 64 == 0 && C <= 1024 && B > 0 && B <= 65535 && H > 0 && W > 0, ACX_ERR_ARG, "head: unsupported shape");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  dim3 pgrid(C / 64, B);
  if (act_dtype == ACX_BF16)
    ACX_CUDA(launch_pdl(valid ? head_pool_kernel<bf16, true> : head_pool_kernel<bf16>, pgrid, dim3(256), 0, st, 1, PDL_SMALL,
                        reinterpret_cast<const bf16*>(x), pooled, H, W, C, valid));
  else
    ACX_CUDA(launch_pdl(valid ? head_pool_kernel<float, true> : head_pool_kernel<float>, pgrid, dim3(256), 0, st, 1, PDL_SMALL,
                        reinterpret_cast<const float*>(x), pooled, H, W, C, valid));
  dim3 fgrid(B, n_cls > 0 ? 8 : 1);
  ACX_CUDA(launch_pdl(head_ln_fc_kernel, fgrid, dim3(256), C * sizeof(float), st, 1, PDL_SMALL, pooled, ln_w, ln_b, fc_w, fc_b, scene, logits,
                      probs, C, n_cls));
  return ACX_OK;
}

int acx_head(const void* x, const float* ln_w, const float* ln_b, const float* fc_w, const float* fc_b, float* pooled,
             float* scene, float* logits, float* probs, int B, int H, int W, int C, int n_cls, int act_dtype,
             void* stream) {
  return head_impl(x, ln_w, ln_b, fc_w, fc_b, pooled, scene, logits, probs, B, H, W, C, n_cls, act_dtype, nullptr, stream);
}

int acx_head_ragged(const void* x, const float* ln_w, const float* ln_b, const float* fc_w, const float* fc_b, float* pooled,
                    float* scene, float* logits, float* probs, int B, int H, int W, int C, int n_cls, int act_dtype,
                    const int32_t* valid, void* stream) {
  ACX_CHECK(valid, ACX_ERR_ARG, "head_ragged: null valid-length array");
  return head_impl(x, ln_w, ln_b, fc_w, fc_b, pooled, scene, logits, probs, B, H, W, C, n_cls, act_dtype, valid, stream);
}

static int nhwc_to_nchw_impl(const void* x, float* out, int B, int H, int W, int C, int act_dtype, const int32_t* valid,
                             void* stream) {
  ACX_CHECK(x && out && B > 0 && B <= 65535, ACX_ERR_ARG, "nhwc_to_nchw: bad arguments");
  ACX_CHECK(!valid || (H > 0 && W > 0), ACX_ERR_ARG, "nhwc_to_nchw: H=%d W=%d must be positive", H, W);
  const int HW = H * W;
  dim3 grid(ceil_div(HW, 32), ceil_div(C, 32), B), block(32, 8);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (act_dtype == ACX_BF16)
    ACX_CUDA(launch_pdl(valid ? nhwc_to_nchw_kernel<bf16, true> : nhwc_to_nchw_kernel<bf16>, grid, block, 0, st, 1, PDL_SMALL,
                        reinterpret_cast<const bf16*>(x), out, HW, C, W, valid));
  else
    ACX_CUDA(launch_pdl(valid ? nhwc_to_nchw_kernel<float, true> : nhwc_to_nchw_kernel<float>, grid, block, 0, st, 1, PDL_SMALL,
                        reinterpret_cast<const float*>(x), out, HW, C, W, valid));
  return ACX_OK;
}

int acx_nhwc_to_nchw_f32(const void* x, float* out, int B, int H, int W, int C, int act_dtype, void* stream) {
  return nhwc_to_nchw_impl(x, out, B, H, W, C, act_dtype, nullptr, stream);
}

int acx_nhwc_to_nchw_f32_ragged(const void* x, float* out, int B, int H, int W, int C, int act_dtype, const int32_t* valid,
                                void* stream) {
  ACX_CHECK(valid, ACX_ERR_ARG, "nhwc_to_nchw_ragged: null valid-length array");
  return nhwc_to_nchw_impl(x, out, B, H, W, C, act_dtype, valid, stream);
}

int acx_resample_fit(const float* x, int ld_in, const float* taps, float* out, int ld_out, int B, int L_in, int orig,
                     int newf, int width, int n_out, void* stream) {
  ACX_CHECK(x && taps && out, ACX_ERR_ARG, "resample_fit: null pointer");
  ACX_CHECK(B > 0 && B <= 65535 && L_in > 0 && n_out > 0, ACX_ERR_ARG, "resample_fit: bad sizes B=%d L_in=%d n_out=%d", B,
            L_in, n_out);
  ACX_CHECK(orig > 0 && newf > 0 && width > 0, ACX_ERR_ARG, "resample_fit: bad rates %d -> %d (width %d)", orig, newf,
            width);
  ACX_CHECK(ld_in >= L_in && ld_out >= n_out, ACX_ERR_ARG, "resample_fit: row pitch smaller than row length");
  const long long target = ((long long)newf * L_in + orig - 1) / orig;
  dim3 grid(ceil_div(n_out, 256), B);
  resample_fit_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(x, ld_in, taps, out, ld_out, L_in, orig,
                                                                                newf, width, n_out, target);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

}  // extern "C"

static int resample_tiling_checked(int orig, int newf, int width, ResampleTiling* t) {
  ACX_CHECK(orig > 0 && newf > 0 && width > 0, ACX_ERR_ARG, "resample_segments: bad rates %d -> %d (width %d)", orig,
            newf, width);
  *t = resample_tiling(orig, newf, width);
  ACX_CHECK(t->smem <= RS_MAX_SMEM, ACX_ERR_UNSUPPORTED,
            "resample_segments: rate ratio %d/%d (K=%lld taps) needs %lld bytes of shared memory per tile, over %d",
            orig, newf, 2LL * width + orig, t->smem, RS_MAX_SMEM);
  return ACX_OK;
}

template <typename TIn, bool STREAM = false>
static int resample_segments_impl(const TIn* x, long long x_len, const long long* seg, int S, const long long* tile_start,
                                  long long n_tiles, const float* taps, int orig, int newf, int width, float* out,
                                  long long out_len, void* stream) {
  const char* what = STREAM ? "resample_stream" : "resample_segments";
  ACX_CHECK(x && seg && tile_start && taps && out, ACX_ERR_ARG, "%s: null pointer", what);
  ACX_CHECK(S >= 1 && x_len >= 1 && out_len >= 1, ACX_ERR_ARG, "%s: bad sizes S=%d x_len=%lld out_len=%lld", what, S,
            x_len, out_len);
  ACX_CHECK(n_tiles >= 1 && n_tiles <= 0x7fffffffLL, ACX_ERR_ARG, "%s: n_tiles=%lld out of [1, 2^31)", what, n_tiles);
  ResampleTiling t;
  const int rc = resample_tiling_checked(orig, newf, width, &t);
  if (rc != ACX_OK) return rc;
  auto kern = resample_segments_kernel<TIn, STREAM>;
  ACX_SET_MAX_SMEM(kern, RS_MAX_SMEM);
  kern<<<(unsigned)n_tiles, RS_THREADS, (size_t)t.smem, reinterpret_cast<cudaStream_t>(stream)>>>(
      x, x_len, seg, tile_start, S, taps, orig, newf, width, t.P, t.F, t.G, out, out_len);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

extern "C" {

int acx_resample_segments_tiling(int orig, int newf, int width, int* tile_frames_host, int* phase_groups_host) {
  ACX_CHECK(tile_frames_host && phase_groups_host, ACX_ERR_ARG, "resample_segments_tiling: null pointer");
  ResampleTiling t;
  const int rc = resample_tiling_checked(orig, newf, width, &t);
  if (rc != ACX_OK) return rc;
  *tile_frames_host = t.F;
  *phase_groups_host = t.G;
  return ACX_OK;
}

int acx_resample_segments(const float* x, long long x_len, const long long* seg, int S, const long long* tile_start,
                          long long n_tiles, const float* taps, int orig, int newf, int width, float* out,
                          long long out_len, void* stream) {
  return resample_segments_impl<float>(x, x_len, seg, S, tile_start, n_tiles, taps, orig, newf, width, out, out_len,
                                       stream);
}

int acx_resample_segments_pcm16(const int16_t* x, long long x_len, const long long* seg, int S,
                                const long long* tile_start, long long n_tiles, const float* taps, int orig, int newf,
                                int width, float* out, long long out_len, void* stream) {
  return resample_segments_impl<int16_t>(x, x_len, seg, S, tile_start, n_tiles, taps, orig, newf, width, out, out_len,
                                         stream);
}

int acx_resample_stream(const float* x, long long x_len, const long long* table, int S, const long long* tile_start,
                        long long n_tiles, const float* taps, int orig, int newf, int width, float* out, long long out_len,
                        void* stream) {
  return resample_segments_impl<float, true>(x, x_len, table, S, tile_start, n_tiles, taps, orig, newf, width, out,
                                             out_len, stream);
}

}  // extern "C"

template <typename TIn>
static int stream_append_impl(const TIn* src, long long src_len, const long long* table, int S, float* ring,
                              long long ring_len, void* stream) {
  ACX_CHECK(src && table && ring, ACX_ERR_ARG, "stream_append: null pointer");
  ACX_CHECK(S >= 1 && src_len >= 1 && src_len <= 0x7fffffffLL * 256 && ring_len >= 1, ACX_ERR_ARG,
            "stream_append: bad sizes S=%d src_len=%lld ring_len=%lld", S, src_len, ring_len);
  stream_append_kernel<TIn><<<(unsigned)((src_len + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      src, src_len, table, S, ring, ring_len);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

extern "C" {

int acx_stream_append(const float* src, long long src_len, const long long* table, int S, float* ring, long long ring_len,
                      void* stream) {
  return stream_append_impl<float>(src, src_len, table, S, ring, ring_len, stream);
}

int acx_stream_append_pcm16(const int16_t* src, long long src_len, const long long* table, int S, float* ring,
                            long long ring_len, void* stream) {
  return stream_append_impl<int16_t>(src, src_len, table, S, ring, ring_len, stream);
}

}  // extern "C"
