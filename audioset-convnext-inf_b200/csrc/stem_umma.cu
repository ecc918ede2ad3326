// Stem on the tensor cores (bf16 mode): Conv2d(1, 96, 4x4, stride 4, pad (4, 0)) + channels_first LayerNorm(96)
// (reference convnext.py:688-691 + :227) as a 128 x 96 x 16 GEMM per 128 output pixels.
//
// The CUDA-core version (kernels_bw.cu::stem_kernel, kept for the fp32-accurate mode) spends 1536 FMAs per pixel on the
// FP32 pipe: 1.4 GFMA per 64 clips, ~145 us, 4x its HBM time.  Here a CTA (128 threads = 128 TMEM lanes = 128 pixels)
//   1. gathers each pixel's 4 x 4 fp32 patch (four float4 loads), splits it into bf16 hi + lo (16 operand bits) and
//      writes one 32-byte K-major row per pixel into 128B-swizzled A tiles;
//   2. one thread issues  D = Ahi.Whi + Alo.Whi + Ahi.Wlo  (tcgen05.mma M=128, N=96, K=16, fp32 accumulate in TMEM; the
//      fp32 conv weight is split the same way once per CTA), i.e. the product carries ~16 mantissa bits like the
//      split-precision front end, not bf16's 8;
//   3. every thread reads ITS pixel's 96 channels back with tcgen05.ld, adds the bias, does the LayerNorm entirely in
//      registers (two-pass variance, no cross-thread traffic), packs bf16 and stages the row in smem (the A tiles'
//      space: the MMAs have completed), from where the warp's 32 contiguous rows are stored with coalesced 16-byte writes.
// The next tile's patch is requested before the epilogue, and 4 CTAs share an SM (47 KB of smem and 128 TMEM columns
// each), so HBM latency, MMA and epilogue of different tiles overlap.
#include "common.cuh"
#include "ptx.cuh"

namespace acx {

struct StemCfg {
  static constexpr int CO = 96, BM = 128;
  static constexpr int A_TILE = BM * 128;              // 128 rows x 128 B (only 32 B per row carry K = 16)
  static constexpr int W_TILE = CO * 64;               // 96 rows x 64 B, SWIZZLE_64B (the 16 taps fill half a row)
  static constexpr int OFF_AHI = 0;
  static constexpr int OFF_ALO = OFF_AHI + A_TILE;
  static constexpr int OFF_WHI = OFF_ALO + A_TILE;     // 32 KB
  static constexpr int OFF_WLO = OFF_WHI + W_TILE;
  static constexpr int OFF_VEC = OFF_WLO + W_TILE;     // bias, ln_w, ln_b: 3 x 96 fp32
  static constexpr int OFF_BAR = OFF_VEC + 3 * CO * 4;
  static constexpr int SMEM_BYTES = OFF_BAR + 64 + 1024 /*align*/;
  static constexpr int ROW_BYTES = CO * 2;             // 192
  static constexpr int ROW_PITCH = ROW_BYTES + 16;     // conflict-free 16-byte row writes
  static constexpr int TMEM_COLS = 128;
  static_assert(4 * 32 * ROW_PITCH <= 2 * A_TILE, "output staging aliases the A tiles");
};

__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat16 ah = __float2bfloat16_rn(a), bh = __float2bfloat16_rn(b);
  const __nv_bfloat16 al = __float2bfloat16_rn(a - __bfloat162float(ah)), bl = __float2bfloat16_rn(b - __bfloat162float(bh));
  hi = (uint32_t)__bfloat16_as_ushort(ah) | ((uint32_t)__bfloat16_as_ushort(bh) << 16);
  lo = (uint32_t)__bfloat16_as_ushort(al) | ((uint32_t)__bfloat16_as_ushort(bl) << 16);
}

// RAG: clip b has valid[b] frames (clamped to [0, Tn]); later rows are read as the conv's zero padding.
template <bool RAG = false>
__global__ void __launch_bounds__(128, 4)
    stem_umma_kernel(const float* __restrict__ logmel, const float* __restrict__ w, const float* __restrict__ bias,
                     const float* __restrict__ ln_w, const float* __restrict__ ln_b, bf16* __restrict__ out, int Tn,
                     int n_mels, int H0, int W0, long long total, int gp, const int32_t* __restrict__ valid) {
  using Cfg = StemCfg;
  constexpr int CO = Cfg::CO;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* svec = reinterpret_cast<float*>(smem + Cfg::OFF_VEC);
  uint64_t* mma_done = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_done + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  // ---- once per CTA: split weights (K-major rows of 16 taps, 64B swizzle), vectors, barrier, TMEM --------------------
  if (tid < CO) {
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int k = 0; k < 16; k += 2) split_bf16x2(w[k * CO + tid], w[(k + 1) * CO + tid], hi[k / 2], lo[k / 2]);
    const int sw = (tid >> 1) & 3;                       // SWIZZLE_64B: 16-byte chunk j of row r sits at j ^ ((r >> 1) & 3)
    uint8_t* rh = smem + Cfg::OFF_WHI + tid * 64;
    uint8_t* rl = smem + Cfg::OFF_WLO + tid * 64;
    *reinterpret_cast<uint4*>(rh + ((0 ^ sw) << 4)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(rh + ((1 ^ sw) << 4)) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
    *reinterpret_cast<uint4*>(rl + ((0 ^ sw) << 4)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    *reinterpret_cast<uint4*>(rl + ((1 ^ sw) << 4)) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
    svec[tid] = bias[tid];
    svec[CO + tid] = ln_w[tid];
    svec[2 * CO + tid] = ln_b[tid];
  }
  if (warp == 1 && ptx::elect_one()) {
    ptx::mbar_init(mma_done, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 0) {
    ptx::tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::fence_proxy_async_smem();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_d = *tmem_slot;
  pdl_trigger();       // programmatic dependent launch (common.cuh): weights split, TMEM allocated
  pdl_wait();          // the log-mel is the front end's output
  const uint32_t lane_taddr = tmem_d + (static_cast<uint32_t>(warp * 32) << 16);
  const uint32_t sbase = ptx::smem_u32(smem);
  const uint64_t dAhi = ptx::umma_desc_sw128_kmajor(sbase + Cfg::OFF_AHI);
  const uint64_t dAlo = ptx::umma_desc_sw128_kmajor(sbase + Cfg::OFF_ALO);
  const uint64_t dWhi = ptx::umma_desc_sw64_kmajor(sbase + Cfg::OFF_WHI);
  const uint64_t dWlo = ptx::umma_desc_sw64_kmajor(sbase + Cfg::OFF_WLO);
  constexpr uint32_t idesc = ptx::umma_idesc_bf16(Cfg::BM, CO);

  const long long num_tiles = (total + Cfg::BM - 1) / Cfg::BM;
  auto load_patch = [&](long long tile, float4 (&v)[4]) {
    const long long pix = tile * Cfg::BM + tid;
    const bool ok = tile < num_tiles && pix < total;
    const long long pp = ok ? pix : 0;
    const int ox = (int)(pp % W0);
    const int oy = (int)((pp / W0) % H0);
    const long long b = pp / ((long long)W0 * H0);
    const int Tb = RAG ? min(max(__ldg(valid + b), 0), Tn) : Tn;
#pragma unroll
    for (int ky = 0; ky < 4; ++ky) {
      const int t = oy * 4 - 4 + ky;                           // 4 rows of zero padding in time (pad = (4, 0))
      v[ky] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ok && t >= 0 && t < Tb) v[ky] = __ldg(reinterpret_cast<const float4*>(logmel + ((size_t)b * Tn + t) * n_mels + ox * 4));
    }
  };

  float4 patch[4];
  load_patch(blockIdx.x, patch);
  uint32_t it = 0;
  for (long long tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
    // ---- 1. this pixel's K-major row (16 taps = 32 B) into the hi and lo A tiles ---------------------------------
    {
      uint32_t hi[8], lo[8];
#pragma unroll
      for (int ky = 0; ky < 4; ++ky) {
        split_bf16x2(patch[ky].x, patch[ky].y, hi[2 * ky], lo[2 * ky]);
        split_bf16x2(patch[ky].z, patch[ky].w, hi[2 * ky + 1], lo[2 * ky + 1]);
      }
      const int sw = tid & 7;
      uint8_t* rh = smem + Cfg::OFF_AHI + tid * 128;
      uint8_t* rl = smem + Cfg::OFF_ALO + tid * 128;
      *reinterpret_cast<uint4*>(rh + ((0 ^ sw) << 4)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
      *reinterpret_cast<uint4*>(rh + ((1 ^ sw) << 4)) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
      *reinterpret_cast<uint4*>(rl + ((0 ^ sw) << 4)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      *reinterpret_cast<uint4*>(rl + ((1 ^ sw) << 4)) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
    }
    ptx::fence_proxy_async_smem();
    ptx::tc_fence_before();
    __syncthreads();
    // ---- 2. D = Ahi.Whi + Alo.Whi + Ahi.Wlo ----------------------------------------------------------------------
    if (warp == 0 && ptx::elect_one()) {
      ptx::tc_fence_after();
      ptx::umma_bf16(tmem_d, dAhi, dWhi, idesc, 0u);
      ptx::umma_bf16(tmem_d, dAlo, dWhi, idesc, 1u);
      ptx::umma_bf16(tmem_d, dAhi, dWlo, idesc, 1u);
      ptx::umma_commit(mma_done);
    }
    load_patch(tile + gridDim.x, patch);                         // next tile's patch: its HBM latency hides below
    ptx::mbar_wait(mma_done, it & 1);
    ptx::tc_fence_after();
    // ---- 3. bias + LayerNorm(96) in registers ---------------------------------------------------------------------
    uint32_t r0[32], r1[32], r2[32];
    ptx::tmem_ld_32x32b_x32(lane_taddr, r0);
    ptx::tmem_ld_32x32b_x32(lane_taddr + 32, r1);
    ptx::tmem_ld_32x32b_x32(lane_taddr + 64, r2);
    ptx::tmem_ld_wait();
    float v[CO];
    float sum = 0.f;
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      v[c] = __uint_as_float(r0[c]) + svec[c];
      v[32 + c] = __uint_as_float(r1[c]) + svec[32 + c];
      v[64 + c] = __uint_as_float(r2[c]) + svec[64 + c];
      sum += v[c] + v[32 + c] + v[64 + c];
    }
    const float mean = sum * (1.0f / CO);
    float sq = 0.f;
#pragma unroll
    for (int c = 0; c < CO; ++c) {
      v[c] -= mean;
      sq = fmaf(v[c], v[c], sq);
    }
    const float rstd = rsqrtf(sq * (1.0f / CO) + 1e-6f);
    // the A tiles are free (the MMAs that read them have completed): stage this warp's 32 x 192 B of output there
    uint8_t* stile = smem + warp * 32 * Cfg::ROW_PITCH;
    uint8_t* myrow = stile + lane * Cfg::ROW_PITCH;
#pragma unroll
    for (int c = 0; c < CO; c += 8) {
      uint4 q;
      q.x = Pair<bf16>::pack(v[c + 0] * rstd * svec[CO + c + 0] + svec[2 * CO + c + 0], v[c + 1] * rstd * svec[CO + c + 1] + svec[2 * CO + c + 1]);
      q.y = Pair<bf16>::pack(v[c + 2] * rstd * svec[CO + c + 2] + svec[2 * CO + c + 2], v[c + 3] * rstd * svec[CO + c + 3] + svec[2 * CO + c + 3]);
      q.z = Pair<bf16>::pack(v[c + 4] * rstd * svec[CO + c + 4] + svec[2 * CO + c + 4], v[c + 5] * rstd * svec[CO + c + 5] + svec[2 * CO + c + 5]);
      q.w = Pair<bf16>::pack(v[c + 6] * rstd * svec[CO + c + 6] + svec[2 * CO + c + 6], v[c + 7] * rstd * svec[CO + c + 7] + svec[2 * CO + c + 7]);
      *reinterpret_cast<uint4*>(myrow + c * 2) = q;
    }
    __syncwarp();
    const long long warp_pix0 = tile * Cfg::BM + warp * 32;
    const long long left = total - warp_pix0;
    const int n_valid = left < 0 ? 0 : (left < 32 ? (int)left : 32);
    uint8_t* gdst = reinterpret_cast<uint8_t*>(out) + (size_t)warp_pix0 * Cfg::ROW_BYTES;
    constexpr int PIECES = Cfg::ROW_BYTES / 16;
    if (gp) {
      // group-planar output [12][Mp][8] (the layout the tensor-core depthwise conv of stage 0 reads): piece pc of this
      // warp's rows is a contiguous 16 B x n_valid run of plane pc
      const long long mp = (total + 127) / 128 * 128;
      for (int i = lane; i < n_valid * PIECES; i += 32) {
        const int pc = i / n_valid, r = i - pc * n_valid;
        *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(out) + ((size_t)pc * mp + warp_pix0 + r) * 16) =
            *reinterpret_cast<const uint4*>(stile + r * Cfg::ROW_PITCH + pc * 16);
      }
    } else
    for (int i = lane; i < n_valid * PIECES; i += 32) {
      const int r = i / PIECES, pc = i % PIECES;
      *reinterpret_cast<uint4*>(gdst + (size_t)r * Cfg::ROW_BYTES + pc * 16) =
          *reinterpret_cast<const uint4*>(stile + r * Cfg::ROW_PITCH + pc * 16);
    }
    // the next iteration overwrites the A tiles (= this staging area) and D: every warp must be done with both
    ptx::tc_fence_before();
    __syncthreads();
  }
  if (warp == 0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_d, Cfg::TMEM_COLS);
  }
}

int launch_stem_umma(const float* logmel, const float* w, const float* bias, const float* ln_w, const float* ln_b,
                     void* out, int B, int T, int n_mels, int gp, const int32_t* valid, cudaStream_t st) {
  using Cfg = StemCfg;
  const int H0 = (T + 4) / 4 + 1, W0 = n_mels / 4;
  const long long total = (long long)B * H0 * W0;
  auto kern = valid ? stem_umma_kernel<true> : stem_umma_kernel<false>;
  if (valid) ACX_SET_MAX_SMEM(stem_umma_kernel<true>, Cfg::SMEM_BYTES);
  else ACX_SET_MAX_SMEM(stem_umma_kernel<false>, Cfg::SMEM_BYTES);
  int dev = 0, sms = 0;
  ACX_CUDA(cudaGetDevice(&dev));
  ACX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const long long tiles = (total + Cfg::BM - 1) / Cfg::BM;
  const long long want = 4LL * sms;                              // 4 resident CTAs per SM (4 x 128 TMEM columns)
  const int grid = (int)(tiles < want ? tiles : want);
  ACX_CUDA(launch_pdl(kern, dim3(grid), dim3(128), Cfg::SMEM_BYTES, st, 1, PDL_SMALL, logmel, w, bias, ln_w, ln_b,
                      reinterpret_cast<bf16*>(out), T, n_mels, H0, W0, total, gp, valid));
  return ACX_OK;
}

}  // namespace acx
