// Fused front end on FOLDED frames: the real-input symmetry of the windowed DFT halves the tensor-core work of
// frontend_fused.cu.  Replaces torchlibrosa Spectrogram + LogmelFilterBank + bn0 (reference convnext.py:298-306).
//
// The STFT rows the checkpoint carries are W_re[k, n] = w[n] cos(2 pi k n / N), W_im[k, n] = -w[n] sin(2 pi k n / N) with a
// periodic Hann window (w[0] = 0, w[N - n] = w[n]):  W_re[k, N - n] = W_re[k, n],  W_im[k, N - n] = -W_im[k, n].  With
//     E[0] = x[N/2],  E[j] = x[j] + x[N - j],  O[0] = 0,  O[j] = x[j] - x[N - j]        (j = 1 .. N/2 - 1)
// a frame's spectrum is   re[k] = sum_j E[j] W_re[k, j'],   im[k] = sum_j O[j] W_im[k, j]     (j' = N/2 for j = 0, else j):
// two K = 512 products instead of one K = 1024 product over [re | im].  The engine checks the symmetry of the LOADED
// weights (engine.fold_dft_weights) and keeps the dense kernel when it does not hold.
//
//   acx_frame_fold      waveform (fp32 or int16 PCM) -> F[b, t, 0..511] = E, F[b, t, 512..1023] = O of frame t (reflect
//                       padding as torchlibrosa: center=True), scaled by 2^ACX_FE_SCALE_LOG2 and split into fp16 hi / lo.
//                       The fold happens in fp32 BEFORE the split, so the operand precision is that of the dense path.
//   acx_frontend_folded one CTA = 128 consecutive frames of one clip; bins in PAIRS of 64-bin chunks (p = 0 .. ceil(n / 2)):
//       GEMM_re(p): D_re[128 x 128] = E[128 x 512] . Wre_p[128 x 512]^T      (columns: re of chunk 2p | re of chunk 2p + 1)
//       GEMM_im(p): D_im[128 x 128] = O[128 x 512] . Wim_p[128 x 512]^T
//     (N = 128 per MMA keeps the operand streaming of an MMA -- 4 KB of A + 4 KB of B per K step at 128 B/clk -- balanced
//     against its math; splitting re and im of ONE chunk into two N = 64 MMAs would only save a quarter.)  Split precision x3
//     as in the dense kernel.  The epilogue warps read re(p) into registers as soon as it is complete -- which frees D_re
//     for GEMM_re(p + 1) while GEMM_im(p) still runs -- then per chunk: P = re^2 + im^2 -> bf16 hi / lo -> smem ->
//       GEMM2(c):   D2[128 x 224] += P[128 x 64] . mel_c[224 x 64]^T, and after the last chunk the log-mel epilogue.
// Warps: 0 = TMA ring producer, 1 = MMA issuer, 2 = TMEM alloc, 3 = mel-chunk TMA producer, 4..11 = epilogue.
#include "common.cuh"
#include "ptx.cuh"
#include "tmap.cuh"

namespace acx {

struct FfArgs {
  float* out;
  const float* bn_scale;
  const float* bn_shift;
  int T, n_chunks, tiles_per_clip, n_mels;
};

namespace ff {
constexpr int BM = 128, BK = 64, NKH = 8 /* K blocks per half: 512 / 64 */;
constexpr int TILE = BM * BK * 2;            // 16 KB: one 128 x 64 two-byte operand tile
constexpr int STAGE = 4 * TILE;              // Ahi, Alo, Bhi, Blo
constexpr int STAGES = 2;
constexpr int MEL_ROWS = 224;
constexpr int MEL_TILE = MEL_ROWS * BK * 2;  // 28 KB
constexpr int OFF_P = STAGES * STAGE;        // P_hi, P_lo
constexpr int OFF_MEL = OFF_P + 2 * TILE;    // mel_hi, mel_lo
constexpr int OFF_BAR = OFF_MEL + 2 * MEL_TILE;
constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;
constexpr int NEPI = 8;
constexpr int THREADS = 128 + 32 * NEPI;
constexpr int D1_COLS = 128, D2_COL0 = 256, TMEM_COLS = 512;
static_assert(SMEM_BYTES <= 227 * 1024, "front-end smem budget");
}  // namespace ff

__global__ void __launch_bounds__(ff::THREADS, 1)
    frontend_folded_kernel(const __grid_constant__ CUtensorMap tmFHi, const __grid_constant__ CUtensorMap tmFLo,
                           const __grid_constant__ CUtensorMap tmWHi, const __grid_constant__ CUtensorMap tmWLo,
                           const __grid_constant__ CUtensorMap tmMelHi, const __grid_constant__ CUtensorMap tmMelLo,
                           FfArgs a) {
  using namespace ff;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* d1_full = empty_bar + STAGES;      // [0] = D_re complete, [1] = D_im complete
  uint64_t* d1_empty = d1_full + 2;
  uint64_t* p_full = d1_empty + 2;
  uint64_t* g2_done = p_full + 1;
  uint64_t* mel_full = g2_done + 1;
  uint64_t* d2_full = mel_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(d2_full + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int clip = blockIdx.x / a.tiles_per_clip;
  const int t0 = (blockIdx.x % a.tiles_per_clip) * BM;
  const int n_pairs = (a.n_chunks + 1) >> 1;

  if (warp == 0 && ptx::elect_one()) {
    ptx::prefetch_tensormap(&tmFHi);
    ptx::prefetch_tensormap(&tmFLo);
    ptx::prefetch_tensormap(&tmWHi);
    ptx::prefetch_tensormap(&tmWLo);
    ptx::prefetch_tensormap(&tmMelHi);
    ptx::prefetch_tensormap(&tmMelLo);
  }
  if (warp == 1 && ptx::elect_one()) {
    for (int s = 0; s < STAGES; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&d1_full[i], 1);
      ptx::mbar_init(&d1_empty[i], NEPI);
    }
    ptx::mbar_init(p_full, NEPI);
    ptx::mbar_init(g2_done, 1);
    ptx::mbar_init(mel_full, 1);
    ptx::mbar_init(d2_full, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_trigger();       // programmatic dependent launch (common.cuh): resources acquired, dependents may be scheduled
  pdl_wait();          // the folded frames are acx_frame_fold's output
  uint8_t* sP = smem + OFF_P;
  uint8_t* sMel = smem + OFF_MEL;

  if (warp == 0) {
    // ===================== ring producer: folded frames (hi, lo) + DFT rows of the pair (hi, lo) =====================
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int p = 0; p < n_pairs; ++p) {
        for (int kb = 0; kb < 2 * NKH; ++kb) {           // kb < 8: E x re rows, kb >= 8: O x im rows
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* s = smem + stage * STAGE;
          ptx::mbar_arrive_expect_tx(&full_bar[stage], STAGE);
          ptx::tma_load_3d(s, &tmFHi, &full_bar[stage], kb * BK, t0, clip);
          ptx::tma_load_3d(s + TILE, &tmFLo, &full_bar[stage], kb * BK, t0, clip);
          ptx::tma_load_2d(s + 2 * TILE, &tmWHi, &full_bar[stage], (kb & (NKH - 1)) * BK, p * 256 + (kb >> 3) * 128);
          ptx::tma_load_2d(s + 3 * TILE, &tmWLo, &full_bar[stage], (kb & (NKH - 1)) * BK, p * 256 + (kb >> 3) * 128);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 3) {
    // ===================== mel-chunk producer ============================================================
    if (ptx::elect_one()) {
      for (int c = 0; c < a.n_chunks; ++c) {
        if (c > 0) ptx::mbar_wait(g2_done, (c - 1) & 1);  // GEMM2(c-1) finished reading the mel buffer
        ptx::mbar_arrive_expect_tx(mel_full, 2 * MEL_TILE);
        ptx::tma_load_2d(sMel, &tmMelHi, mel_full, 0, c * 256);
        ptx::tma_load_2d(sMel + MEL_TILE, &tmMelLo, mel_full, 0, c * 256);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer ====================================================================
    if (ptx::elect_one()) {
      constexpr uint32_t idesc128 = ptx::umma_idesc_f16(BM, 128);      // fp16 x fp16 -> fp32 (scaled split operands)
      constexpr uint32_t idesc64 = ptx::umma_idesc_f16(BM, 64);        // last pair of an odd chunk count: one chunk only
      constexpr uint32_t idesc2 = ptx::umma_idesc_bf16(BM, MEL_ROWS);
      const uint32_t d2 = tmem_base + D2_COL0;
      const uint64_t dPhi = ptx::umma_desc_sw128_kmajor(ptx::smem_u32(sP));
      const uint64_t dPlo = ptx::umma_desc_sw128_kmajor(ptx::smem_u32(sP + TILE));
      const uint64_t dMhi = ptx::umma_desc_sw128_kmajor(ptx::smem_u32(sMel));
      const uint64_t dMlo = ptx::umma_desc_sw128_kmajor(ptx::smem_u32(sMel + MEL_TILE));
      auto gemm2 = [&](int cc) {
        ptx::mbar_wait(p_full, cc & 1);
        ptx::mbar_wait(mel_full, cc & 1);
        ptx::tc_fence_after();
#pragma unroll
        for (int k = 0; k < BK / 16; ++k) {
          ptx::umma_bf16(d2, dPhi + 2 * k, dMhi + 2 * k, idesc2, (cc | k) != 0 ? 1u : 0u);
          ptx::umma_bf16(d2, dPhi + 2 * k, dMlo + 2 * k, idesc2, 1u);
          ptx::umma_bf16(d2, dPlo + 2 * k, dMhi + 2 * k, idesc2, 1u);
        }
        ptx::umma_commit(g2_done);
      };
      int stage = 0;
      uint32_t phase = 0;
      for (int p = 0; p < n_pairs; ++p) {
        const uint32_t idesc1 = (2 * p + 1 < a.n_chunks) ? idesc128 : idesc64;
        for (int half = 0; half < 2; ++half) {            // 0: D_re = E . Wre^T, 1: D_im = O . Wim^T
          ptx::mbar_wait(&d1_empty[half], (p & 1) ^ 1);
          ptx::tc_fence_after();
          const uint32_t d1 = tmem_base + half * D1_COLS;
          for (int kb = 0; kb < NKH; ++kb) {
            ptx::mbar_wait(&full_bar[stage], phase);
            ptx::tc_fence_after();
            const uint32_t s = ptx::smem_u32(smem + stage * STAGE);
            const uint64_t dAhi = ptx::umma_desc_sw128_kmajor(s);
            const uint64_t dAlo = ptx::umma_desc_sw128_kmajor(s + TILE);
            const uint64_t dBhi = ptx::umma_desc_sw128_kmajor(s + 2 * TILE);
            const uint64_t dBlo = ptx::umma_desc_sw128_kmajor(s + 3 * TILE);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              ptx::umma_bf16(d1, dAhi + 2 * k, dBhi + 2 * k, idesc1, (kb | k) != 0 ? 1u : 0u);
              ptx::umma_bf16(d1, dAhi + 2 * k, dBlo + 2 * k, idesc1, 1u);
              ptx::umma_bf16(d1, dAlo + 2 * k, dBhi + 2 * k, idesc1, 1u);
            }
            ptx::umma_commit(&empty_bar[stage]);
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1;
            }
          }
          ptx::umma_commit(&d1_full[half]);
          // the mel products of the PREVIOUS pair's chunks ride behind this pair's DFT halves: the tensor pipe stays busy
          // while their power tiles are formed
          const int cc = 2 * (p - 1) + half;
          if (p >= 1 && cc < a.n_chunks) gemm2(cc);
        }
      }
      for (int cc = 2 * (n_pairs - 1); cc < a.n_chunks; ++cc) gemm2(cc);
      ptx::umma_commit(d2_full);
    }
  } else if (warp >= 4) {
    // ===================== epilogue ======================================================================
    const int quad = warp & 3;
    const int group = (warp - 4) >> 2;       // bins [32 group, 32 group + 32) of a chunk
    const int row = quad * 32 + lane;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    for (int p = 0; p < n_pairs; ++p) {
      const bool two = 2 * p + 1 < a.n_chunks;
      // re of both chunks as soon as GEMM_re(p) is complete: D_re is free again while GEMM_im(p) still runs
      ptx::mbar_wait(&d1_full[0], p & 1);
      ptx::tc_fence_after();
      uint32_t re[2][32];
      ptx::tmem_ld_32x32b_x32(lane_base + group * 32, re[0]);
      if (two) ptx::tmem_ld_32x32b_x32(lane_base + 64 + group * 32, re[1]);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&d1_empty[0]);
      ptx::mbar_wait(&d1_full[1], p & 1);
      ptx::tc_fence_after();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int c = 2 * p + h;
        if (h == 1 && !two) break;
        uint32_t im[32];
        ptx::tmem_ld_32x32b_x32(lane_base + D1_COLS + h * 64 + group * 32, im);
        ptx::tmem_ld_wait();
        if (h == 1 || !two) {                  // last read of D_im of this pair
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&d1_empty[1]);
        }
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float r0 = __uint_as_float(re[h][2 * j]), i0 = __uint_as_float(im[2 * j]);
          const float r1 = __uint_as_float(re[h][2 * j + 1]), i1 = __uint_as_float(im[2 * j + 1]);
          // operands carried 2^ACX_FE_SCALE_LOG2 each -> the power carries 2^(4 * ACX_FE_SCALE_LOG2): undo it exactly
          constexpr float kUnscale = 1.0f / (float)(1ull << (4 * ACX_FE_SCALE_LOG2));
          const float p0 = fmaf(r0, r0, i0 * i0) * kUnscale, p1 = fmaf(r1, r1, i1 * i1) * kUnscale;
          const __nv_bfloat162 hh = __floats2bfloat162_rn(p0, p1);
          const float2 hf = __bfloat1622float2(hh);
          const __nv_bfloat162 ll = __floats2bfloat162_rn(p0 - hf.x, p1 - hf.y);
          hi[j] = *reinterpret_cast<const uint32_t*>(&hh);
          lo[j] = *reinterpret_cast<const uint32_t*>(&ll);
        }
        if (c >= 1) ptx::mbar_wait(g2_done, (c - 1) & 1);  // GEMM2(c-1) no longer reads P
        // K-major SWIZZLE_128B: row r at r*128 B, 16-byte chunk j stored at chunk (j ^ (r & 7))
        uint8_t* prow_hi = sP + row * 128;
        uint8_t* prow_lo = prow_hi + TILE;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int chunk = ((group * 4 + q) ^ (row & 7)) * 16;
          *reinterpret_cast<uint4*>(prow_hi + chunk) = make_uint4(hi[4 * q], hi[4 * q + 1], hi[4 * q + 2], hi[4 * q + 3]);
          *reinterpret_cast<uint4*>(prow_lo + chunk) = make_uint4(lo[4 * q], lo[4 * q + 1], lo[4 * q + 2], lo[4 * q + 3]);
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(p_full);
      }
    }
    // ---- log-mel epilogue --------------------------------------------------------------------------------
    ptx::mbar_wait(d2_full, 0);
    ptx::tc_fence_after();
    const int t = t0 + row;
    const bool ok = t < a.T;
    float* orow = a.out + ((size_t)clip * a.T + (ok ? t : 0)) * a.n_mels;
    constexpr int COLS = MEL_ROWS / 2;  // 112 per column group
#pragma unroll 1
    for (int c0 = group * COLS; c0 < (group + 1) * COLS; c0 += 16) {
      uint32_t r[16];
      ptx::tmem_ld_32x32b_x16(lane_base + D2_COL0 + c0, r);
      ptx::tmem_ld_wait();
      if (ok) {
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          const float4 sc = __ldg(reinterpret_cast<const float4*>(a.bn_scale + c0 + j));
          const float4 sh = __ldg(reinterpret_cast<const float4*>(a.bn_shift + c0 + j));
          float4 o;
          // 10 log10(x) = 3.0102999566 * log2(x); power_to_db clamps at amin = 1e-10 (reference CX:165)
          o.x = fmaf(3.01029995664f * __log2f(fmaxf(__uint_as_float(r[j + 0]), 1e-10f)), sc.x, sh.x);
          o.y = fmaf(3.01029995664f * __log2f(fmaxf(__uint_as_float(r[j + 1]), 1e-10f)), sc.y, sh.y);
          o.z = fmaf(3.01029995664f * __log2f(fmaxf(__uint_as_float(r[j + 2]), 1e-10f)), sc.z, sh.z);
          o.w = fmaf(3.01029995664f * __log2f(fmaxf(__uint_as_float(r[j + 3]), 1e-10f)), sc.w, sh.w);
          *reinterpret_cast<float4*>(orow + c0 + j) = o;
        }
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, ff::TMEM_COLS);
  }
}

// ---- frame fold ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float ff_sample(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ff_sample(const int16_t* p) { return __fdiv_rn((float)__ldg(p), 32767.0f); }   // utils/utilities.py:226

// RAG: row b is a clip of valid[b] samples (clamped to [n_fft/2 + 1, L]) at row pitch ld_wave, reflected at its own end and
// zero past the reflected range; samples past valid[b] are never read.
// WIN: row b is the window that starts offsets[b] samples into ONE recording of rec_len samples (windows may overlap), of
// L samples or with RAG its own valid[b]; offsets are 64-bit.  Length and offset are clamped to the recording, so no table
// value can make the kernel read outside it.
template <typename TIn, bool RAG = false, bool WIN = false>
__global__ void __launch_bounds__(256) frame_fold_kernel(const TIn* __restrict__ wave, __half* __restrict__ fhi, __half* __restrict__ flo,
                                                         int L, int T, int n_fft, int hop, int ld_wave,
                                                         const int32_t* __restrict__ valid,
                                                         const long long* __restrict__ offsets = nullptr, long long rec_len = 0) {
  // thread = (frame t, four consecutive fold indices j0 .. j0 + 3): 8-byte stores of E and O, hi and lo
  const int b = blockIdx.y;
  const int half_n = n_fft >> 1;
  const int per_frame = half_n >> 2;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)T * per_frame) return;
  const int t = (int)(idx / per_frame), j0 = (int)(idx - (long long)t * per_frame) * 4;
  const TIn* w = wave + (size_t)b * (RAG ? ld_wave : L);
  if (RAG) L = min(max(__ldg(valid + b), half_n + 1), L);
  if (WIN) {
    L = (int)min((long long)L, rec_len);
    w = wave + min(max(__ldg(offsets + b), 0LL), rec_len - L);
  }
  const int s = t * hop - half_n;              // un-padded sample index of frame position 0 (center = True)
  auto x = [&](int m) {
    if ((RAG || WIN) && m >= L + half_n) return 0.f;    // past the padded clip: only frames >= its own frame count get here
    if (m < 0) m = -m;                         // reflect (edge sample not repeated), as F.pad(mode="reflect")
    if (m >= L) m = 2 * (L - 1) - m;
    return ff_sample(w + m);
  };
  constexpr float kScale = (float)(1 << ACX_FE_SCALE_LOG2);
  float e[4], o[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int j = j0 + i;
    if (j == 0) {
      e[i] = x(s + half_n) * kScale;
      o[i] = 0.f;
    } else {
      const float p = x(s + j), q = x(s + n_fft - j);
      e[i] = (p + q) * kScale;
      o[i] = (p - q) * kScale;
    }
  }
  auto split_store = [&](const float (&v)[4], size_t off) {
    uint32_t h[2], l[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const __half2 hh = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
      const float2 hf = __half22float2(hh);
      const __half2 ll = __floats2half2_rn(v[2 * i] - hf.x, v[2 * i + 1] - hf.y);
      h[i] = *reinterpret_cast<const uint32_t*>(&hh);
      l[i] = *reinterpret_cast<const uint32_t*>(&ll);
    }
    *reinterpret_cast<uint2*>(fhi + off) = make_uint2(h[0], h[1]);
    *reinterpret_cast<uint2*>(flo + off) = make_uint2(l[0], l[1]);
  };
  const size_t rowoff = ((size_t)b * T + t) * n_fft;
  split_store(e, rowoff + j0);
  split_store(o, rowoff + half_n + j0);
}

}  // namespace acx

using namespace acx;

static int frame_fold_impl(const void* wave, int pcm16, void* f_hi, void* f_lo, int B, int L, int T, int n_fft, int hop,
                           int ld_wave, const int32_t* valid, void* stream) {
  ACX_CHECK(wave && f_hi && f_lo, ACX_ERR_ARG, "frame_fold: null pointer");
  ACX_CHECK(ld_wave >= L, ACX_ERR_ARG, "frame_fold: row pitch %d < L=%d", ld_wave, L);
  ACX_CHECK(n_fft == 1024 && hop == 320, ACX_ERR_UNSUPPORTED, "frame_fold: built for n_fft=1024, hop=320 (reference convnext.py:161-174)");
  ACX_CHECK(B > 0 && B <= 65535 && L > n_fft / 2 && T == L / hop + 1, ACX_ERR_ARG,
            "frame_fold: bad sizes B=%d L=%d T=%d (reflect padding needs L > n_fft/2, T = L / hop + 1)", B, L, T);
  ACX_CHECK(((reinterpret_cast<uintptr_t>(f_hi) | reinterpret_cast<uintptr_t>(f_lo)) & 15) == 0, ACX_ERR_ARG, "frame_fold: 16-byte alignment");
  const long long work = (long long)T * (n_fft / 8);
  dim3 grid((unsigned)((work + 255) / 256), B);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (pcm16)
    frame_fold_kernel<int16_t><<<grid, 256, 0, st>>>(reinterpret_cast<const int16_t*>(wave), reinterpret_cast<__half*>(f_hi),
                                                     reinterpret_cast<__half*>(f_lo), L, T, n_fft, hop, L, nullptr);
  else if (valid)
    frame_fold_kernel<float, true><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(wave), reinterpret_cast<__half*>(f_hi),
                                                         reinterpret_cast<__half*>(f_lo), L, T, n_fft, hop, ld_wave, valid);
  else
    frame_fold_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(wave), reinterpret_cast<__half*>(f_hi),
                                                   reinterpret_cast<__half*>(f_lo), L, T, n_fft, hop, L, nullptr);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

extern "C" int acx_frame_fold(const float* wave, void* f_hi, void* f_lo, int B, int L, int T, int n_fft, int hop, void* stream) {
  return frame_fold_impl(wave, 0, f_hi, f_lo, B, L, T, n_fft, hop, L, nullptr, stream);
}
extern "C" int acx_frame_fold_ragged(const float* wave, void* f_hi, void* f_lo, int B, int L, int T, int n_fft, int hop, int ld_wave,
                                     const int32_t* valid, void* stream) {
  ACX_CHECK(valid, ACX_ERR_ARG, "frame_fold_ragged: null valid-length array");
  return frame_fold_impl(wave, 0, f_hi, f_lo, B, L, T, n_fft, hop, ld_wave, valid, stream);
}
extern "C" int acx_frame_fold_pcm16(const int16_t* pcm, void* f_hi, void* f_lo, int B, int L, int T, int n_fft, int hop, void* stream) {
  return frame_fold_impl(pcm, 1, f_hi, f_lo, B, L, T, n_fft, hop, L, nullptr, stream);
}

template <typename TIn>
static int frame_fold_windows(const TIn* rec, long long rec_len, const long long* offsets, const int32_t* valid, void* f_hi,
                              void* f_lo, int B, int L, int T, int n_fft, int hop, void* stream) {
  ACX_CHECK(rec && offsets, ACX_ERR_ARG, "frame_fold_windows: null recording or offsets");
  ACX_CHECK(rec_len >= n_fft / 2 + 1, ACX_ERR_ARG, "frame_fold_windows: rec_len=%lld must be > n_fft/2 (reflect padding)",
            rec_len);
  ACX_CHECK(B >= 1, ACX_ERR_ARG, "frame_fold_windows: empty batch B=%d", B);
  ACX_CHECK(f_hi && f_lo, ACX_ERR_ARG, "frame_fold_windows: null pointer");
  ACX_CHECK(n_fft == 1024 && hop == 320, ACX_ERR_UNSUPPORTED, "frame_fold: built for n_fft=1024, hop=320 (reference convnext.py:161-174)");
  ACX_CHECK(B <= 65535 && L > n_fft / 2 && T == L / hop + 1, ACX_ERR_ARG,
            "frame_fold_windows: bad sizes B=%d L=%d T=%d (reflect padding needs L > n_fft/2, T = L / hop + 1)", B, L, T);
  ACX_CHECK(((reinterpret_cast<uintptr_t>(f_hi) | reinterpret_cast<uintptr_t>(f_lo)) & 15) == 0, ACX_ERR_ARG, "frame_fold: 16-byte alignment");
  const long long work = (long long)T * (n_fft / 8);
  dim3 grid((unsigned)((work + 255) / 256), B);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  __half* hi = reinterpret_cast<__half*>(f_hi);
  __half* lo = reinterpret_cast<__half*>(f_lo);
  if (valid)
    frame_fold_kernel<TIn, true, true><<<grid, 256, 0, st>>>(rec, hi, lo, L, T, n_fft, hop, L, valid, offsets, rec_len);
  else
    frame_fold_kernel<TIn, false, true><<<grid, 256, 0, st>>>(rec, hi, lo, L, T, n_fft, hop, L, nullptr, offsets, rec_len);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

extern "C" int acx_frame_fold_windows(const float* rec, long long rec_len, const long long* offsets, const int32_t* valid,
                                      void* f_hi, void* f_lo, int B, int L, int T, int n_fft, int hop, void* stream) {
  return frame_fold_windows<float>(rec, rec_len, offsets, valid, f_hi, f_lo, B, L, T, n_fft, hop, stream);
}
extern "C" int acx_frame_fold_pcm16_windows(const int16_t* rec, long long rec_len, const long long* offsets, const int32_t* valid,
                                            void* f_hi, void* f_lo, int B, int L, int T, int n_fft, int hop, void* stream) {
  return frame_fold_windows<int16_t>(rec, rec_len, offsets, valid, f_hi, f_lo, B, L, T, n_fft, hop, stream);
}

extern "C" int acx_frontend_folded(const void* f_hi, const void* f_lo, const void* w_hi, const void* w_lo, const void* mel_hi,
                                   const void* mel_lo, int n_chunks, const float* bn_scale, const float* bn_shift, float* out,
                                   int B, int T, int n_fft, int n_mels, void* stream) {
  ACX_CHECK(f_hi && f_lo && w_hi && w_lo && mel_hi && mel_lo && bn_scale && bn_shift && out, ACX_ERR_ARG,
            "frontend_folded: null pointer");
  ACX_CHECK(n_fft == 1024 && n_mels == 224, ACX_ERR_UNSUPPORTED,
            "frontend_folded: built for n_fft=1024, 224 mel bins (reference convnext.py:161-174)");
  ACX_CHECK(B > 0 && T > 0 && n_chunks >= 1 && n_chunks <= 9, ACX_ERR_ARG, "frontend_folded: bad sizes");
  const int n_pairs = (n_chunks + 1) / 2;
  CUtensorMap tmFHi, tmFLo, tmWHi, tmWLo, tmMelHi, tmMelLo;
  {
    // (1024 fold slots) x (frame) x (clip): rows past T read as zero, a tile never crosses into the next clip
    cuuint64_t dims[3] = {(cuuint64_t)n_fft, (cuuint64_t)T, (cuuint64_t)B};
    cuuint64_t strides[2] = {(cuuint64_t)n_fft * 2, (cuuint64_t)T * n_fft * 2};
    cuuint32_t box[3] = {64, 128, 1};
    int rc = make_tmap_bf16(&tmFHi, f_hi, 3, dims, strides, box);
    if (rc != ACX_OK) return rc;
    rc = make_tmap_bf16(&tmFLo, f_lo, 3, dims, strides, box);
    if (rc != ACX_OK) return rc;
  }
  int rc = make_tmap_2d_bf16(&tmWHi, w_hi, (uint64_t)n_fft / 2, (uint64_t)n_pairs * 256, (uint64_t)n_fft, 64, 128);
  if (rc != ACX_OK) return rc;
  rc = make_tmap_2d_bf16(&tmWLo, w_lo, (uint64_t)n_fft / 2, (uint64_t)n_pairs * 256, (uint64_t)n_fft, 64, 128);
  if (rc != ACX_OK) return rc;
  rc = make_tmap_2d_bf16(&tmMelHi, mel_hi, 64, (uint64_t)n_chunks * 256, 128, 64, ff::MEL_ROWS);
  if (rc != ACX_OK) return rc;
  rc = make_tmap_2d_bf16(&tmMelLo, mel_lo, 64, (uint64_t)n_chunks * 256, 128, 64, ff::MEL_ROWS);
  if (rc != ACX_OK) return rc;

  ACX_SET_MAX_SMEM(frontend_folded_kernel, ff::SMEM_BYTES);
  FfArgs a;
  a.out = out;
  a.bn_scale = bn_scale;
  a.bn_shift = bn_shift;
  a.T = T;
  a.n_chunks = n_chunks;
  a.tiles_per_clip = ceil_div(T, ff::BM);
  a.n_mels = n_mels;
  const int grid = B * a.tiles_per_clip;
  ACX_CUDA(launch_pdl(frontend_folded_kernel, dim3(grid), dim3(ff::THREADS), ff::SMEM_BYTES, reinterpret_cast<cudaStream_t>(stream), 1,
                      PDL_SMALL, tmFHi, tmFLo, tmWHi, tmWLo, tmMelHi, tmMelLo, a));
  return ACX_OK;
}
