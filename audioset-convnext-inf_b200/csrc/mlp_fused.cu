// Fused ConvNeXt MLP (reference convnext.py:79-86):
//     x[M,C] <- x + gamma * ( GELU( y . W1^T + b1 ) . W2^T + b2 )          W1 (4C, C), W2 (C, 4C), bf16
// One persistent CTA per SM works on 128-row tiles.  The 4C-wide hidden activation never leaves the SM: it is produced
// 128 columns at a time in TMEM (GEMM1 accumulator D1, double buffered), passed through bias+GELU by the epilogue
// warps into a K-major, 128B-swizzled bf16 smem tile (double buffered), and consumed from there as the A operand of
// GEMM2, whose C-wide accumulator D2 stays in TMEM for the whole tile.  HBM traffic per row is 3 C bf16 (y in,
// residual in, x out) instead of the 3 C + 8 C of the two-kernel form.
//
//   warp 0   weight-stream TMA producer: per chunk h the W1 tiles (128 x 64) then the W2 tiles (C x 64) of chunk h-1,
//            in exactly the order the MMA warp consumes them (mbarrier ring)
//   warp 1   MMA issuer (tcgen05.mma cta_group::1 kind::f16): GEMM1(h) is issued BEFORE GEMM2(h-1) so the tensor pipe
//            runs while the epilogue warps turn D1(h-1) into the hidden tile
//   warp 2   TMEM allocator            warp 3   y-tile (A operand) TMA producer
//   warps 4..11   epilogue-1: D1 (TMEM) -> +b1 -> GELU -> bf16 -> swizzled hidden tile in smem, per chunk
//   warps 12..15  epilogue-2: D2 (TMEM) -> +b2, *gamma, +residual (cp.async) -> bf16 -> TMA store, per tile, OFF the
//            critical path (the epilogue-1 warps are already on the next tile)
// TMEM columns: D2 at 0 (C <= 192 -> 256 reserved), D1[0] at 256, D1[1] at 384.
#include <stdlib.h>

#include "common.cuh"
#include "ptx.cuh"
#include "tmap.cuh"

namespace acx {

struct MlpArgs {
  bf16* x;            // residual stream, updated in place
  const float* b1;
  const float* b2;
  const float* gamma;
  int M;
  const float* ln_w;  // optional: channels-last LayerNorm (convnext.py:78) applied to the y tile IN SHARED MEMORY before
  const float* ln_b;  // GEMM1 reads it -- y then holds the raw depthwise-conv output (acx_dwconv_tc); nullptr = y is final
  const float* ln_s;  // FOLD mode: s_j = sum_c W1'[j, c] of the LayerNorm-folded weights W1' = W1 diag(ln_w) (w1 / b1 then
                      // ARE W1' and b1 + W1 ln_b): the kernel only computes per-row statistics of the y tile and applies
                      // the LayerNorm as a rank-1 correction in the GELU epilogue (common.cuh, LnFold)
};

// LayerNorm of one 128-row operand tile in place in shared memory: thread = row, `chunk(j)` = address of the row's j-th
// 16-byte piece (8 channels, already de-swizzled by the caller).  Two sweeps over the row: shifted single-pass statistics
// (shift = the row's first channel, so  E[d^2] - E[d]^2  does not cancel for rows with a large common offset), then
// out = x * (rstd w) + (b - mean rstd w).  fp32 statistics, eps 1e-6, result rounded to bf16 -- the same arithmetic as
// acx_layernorm_rows up to the summation order.  Costs ~8 instructions per channel on the 4 epilogue-2 warps and saves
// the separate LayerNorm pass over HBM (2 x M x C x 2 B).
template <int C, typename ChunkFn>
__device__ __forceinline__ void ln_row_in_smem(ChunkFn chunk, const float* __restrict__ sw, const float* __restrict__ sb) {
  constexpr int NCH = C / 8;
  float shift;
  {
    const uint32_t w0 = *reinterpret_cast<const uint32_t*>(chunk(0));
    shift = __uint_as_float(w0 << 16);
  }
  const float2 sh2 = make_float2(-shift, -shift);
  float2 s = make_float2(0.f, 0.f), q = make_float2(0.f, 0.f);
#pragma unroll 4
  for (int j = 0; j < NCH; ++j) {
    const uint4 v = *reinterpret_cast<const uint4*>(chunk(j));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 d = __fadd2_rn(Pair<bf16>::unpack(w[k]), sh2);
      s = __fadd2_rn(s, d);
      q = __ffma2_rn(d, d, q);
    }
  }
  const float md = (s.x + s.y) * (1.0f / C);                       // mean of the shifted values
  const float var = fmaxf((q.x + q.y) * (1.0f / C) - md * md, 0.f);
  const float rstd = rsqrtf(var + 1e-6f);
  const float nmr = -(md + shift) * rstd;                          // -mean * rstd
  const float2 r2 = make_float2(rstd, rstd), n2 = make_float2(nmr, nmr);
#pragma unroll 2
  for (int j = 0; j < NCH; ++j) {
    uint8_t* pc = chunk(j);
    const uint4 v = *reinterpret_cast<const uint4*>(pc);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 g = *reinterpret_cast<const float2*>(sw + 8 * j + 2 * k);
      const float2 b = *reinterpret_cast<const float2*>(sb + 8 * j + 2 * k);
      const float2 t = __fmul2_rn(r2, g);
      const float2 u = __ffma2_rn(n2, g, b);
      const float2 y = __ffma2_rn(Pair<bf16>::unpack(w[k]), t, u);
      o[k] = Pair<bf16>::pack(y.x, y.y);
    }
    *reinterpret_cast<uint4*>(pc) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// Per-row LayerNorm statistics of an operand tile in shared memory (read only): (rstd, -mean * rstd), same shifted
// single-pass arithmetic as ln_row_in_smem.
template <int C, typename ChunkFn>
__device__ __forceinline__ float2 ln_row_stats_smem(ChunkFn chunk) {
  constexpr int NCH = C / 8;
  const float shift = __uint_as_float(*reinterpret_cast<const uint32_t*>(chunk(0)) << 16);
  const float2 sh2 = make_float2(-shift, -shift);
  float2 s = make_float2(0.f, 0.f), q = make_float2(0.f, 0.f);
#pragma unroll 4
  for (int j = 0; j < NCH; ++j) {
    const uint4 v = *reinterpret_cast<const uint4*>(chunk(j));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 d = __fadd2_rn(Pair<bf16>::unpack(w[k]), sh2);
      s = __fadd2_rn(s, d);
      q = __ffma2_rn(d, d, q);
    }
  }
  const float md = (s.x + s.y) * (1.0f / C);
  const float var = fmaxf((q.x + q.y) * (1.0f / C) - md * md, 0.f);
  const float rstd = rsqrtf(var + 1e-6f);
  return make_float2(rstd, -(md + shift) * rstd);
}

template <int C_>
struct MlpCfg {
  static constexpr int C = C_, HD = 4 * C, BM = 128, NH = 128, BK = 64;
  static constexpr int NC = HD / NH;                  // hidden chunks per tile
  static constexpr int KB1 = (C + BK - 1) / BK;       // k-blocks of GEMM1
  static constexpr int KB2 = NH / BK;                 // k-blocks of GEMM2 per chunk
  static constexpr int A_TILE = BM * BK * 2;          // 16 KB
  static constexpr int A_BUFS = C <= 96 ? 2 : 1;
  static constexpr int W1_TILE = NH * BK * 2;         // 16 KB
  static constexpr int W2_TILE = C * BK * 2;          // 12 / 24 KB
  static constexpr int SLOT = W1_TILE > W2_TILE ? W1_TILE : W2_TILE;
  static constexpr int SLOTS = C <= 96 ? 4 : 3;
  static constexpr int H_TILE = BM * BK * 2;          // one k-block of the hidden tile
  static constexpr int OFF_A = 0;
  static constexpr int OFF_RING = OFF_A + A_BUFS * KB1 * A_TILE;
  static constexpr int OFF_H = OFF_RING + SLOTS * SLOT;
  static constexpr int OFF_STG = OFF_H + 2 * KB2 * H_TILE;
  static constexpr int STG_TILE = 32 * 64;            // 32 rows x 32 bf16, SWIZZLE_64B
  static constexpr int STG_PER_WARP = STG_TILE;       // one tile: residual transpose in, output staging out
  static constexpr int OFF_BAR = OFF_STG + 8 * STG_PER_WARP;
  static constexpr int OFF_VEC = OFF_BAR + 512;       // b1[4C], b2[C], gamma[C], ln_w[C], ln_b[C] staged once per CTA
  static constexpr int SMEM_BYTES = OFF_VEC + (3 * HD + 4 * C) * 4 + 2 * BM * 8 + 1024;   // + {b1, s} interleaved [2 x 4C], row stats [2][128]
  static constexpr int D2_COL = 0, D1_COL = 256, TMEM_COLS = 512;
  static constexpr int OUT_CHUNKS = C / 32;           // 32-column output chunks: 3 / 6
  static constexpr int OUT_G0 = (OUT_CHUNKS + 1) / 2;
  static constexpr int THREADS = 512;                 // 4 control + 8 epilogue-1 + 4 epilogue-2 warps
  static_assert(C % 32 == 0 && C <= 192, "D2 must fit 256 TMEM columns");
  static_assert(SLOT % 1024 == 0 && W2_TILE % 1024 == 0, "swizzle alignment");
  static_assert(SMEM_BYTES <= 227 * 1024, "smem budget");
};

template <int C, bool GP, bool FOLD>   // GP: group-planar y / x, FOLD: rank-1 LayerNorm; see mlp_fused96_kernel
__global__ void __launch_bounds__(512, 1)
    mlp_fused_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmW1,
                     const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmOut, MlpArgs a) {
  using Cfg = MlpCfg<C>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* ring_full = bars;                          // [SLOTS]
  uint64_t* ring_empty = ring_full + Cfg::SLOTS;       // [SLOTS]
  uint64_t* a_full = ring_empty + Cfg::SLOTS;          // [A_BUFS]
  uint64_t* a_empty = a_full + Cfg::A_BUFS;            // [A_BUFS]
  uint64_t* d1_full = a_empty + Cfg::A_BUFS;           // [2]
  uint64_t* d1_empty = d1_full + 2;                    // [2]
  uint64_t* h_full = d1_empty + 2;                     // [2]
  uint64_t* h_empty = h_full + 2;                      // [2]
  uint64_t* d2_full = h_empty + 2;                     // [1]
  uint64_t* d2_empty = d2_full + 1;                    // [1]
  uint64_t* a_ready = d2_empty + 1;                    // [A_BUFS]  y tile normalised in place (LayerNorm mode only)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_ready + Cfg::A_BUFS);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  float* sb1 = reinterpret_cast<float*>(smem + Cfg::OFF_VEC);
  float* sb2 = sb1 + Cfg::HD;
  float* sgamma = sb2 + C;
  float* slnw = sgamma + C;
  float* slnb = slnw + C;
  float* ss1 = slnb + C;                                          // FOLD: {b1[2q], b1[2q+1], s[2q], s[2q+1]} per column pair
  float2* sstat = reinterpret_cast<float2*>(ss1 + 2 * Cfg::HD);   // FOLD: [2][128] (rstd, -mean rstd) per row
  const bool ln = a.ln_w != nullptr;
  for (int i = threadIdx.x; i < Cfg::HD; i += blockDim.x) sb1[i] = a.b1[i];
  if (FOLD)
    for (int i = threadIdx.x; i < Cfg::HD; i += blockDim.x) {
      ss1[4 * (i >> 1) + (i & 1)] = a.b1[i];
      ss1[4 * (i >> 1) + 2 + (i & 1)] = a.ln_s[i];
    }
  if (ln)
    for (int i = threadIdx.x; i < C; i += blockDim.x) {
      slnw[i] = a.ln_w[i];
      slnb[i] = a.ln_b[i];
    }
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    // the hidden tile holds 2 * gelu(.), so  x + gamma (0.5 acc + b2) = x + (0.5 gamma) acc + gamma b2:
    sgamma[i] = 0.5f * a.gamma[i];       // multiplies the GEMM2 accumulator
    sb2[i] = a.gamma[i] * a.b2[i];       // added together with the residual
  }

  if (warp == 0 && ptx::elect_one()) {
    ptx::prefetch_tensormap(&tmY);
    ptx::prefetch_tensormap(&tmW1);
    ptx::prefetch_tensormap(&tmW2);
    ptx::prefetch_tensormap(&tmOut);
  }
  if (warp == 1 && ptx::elect_one()) {
    for (int s = 0; s < Cfg::SLOTS; ++s) {
      ptx::mbar_init(&ring_full[s], 1);
      ptx::mbar_init(&ring_empty[s], 1);
    }
    for (int s = 0; s < Cfg::A_BUFS; ++s) {
      ptx::mbar_init(&a_full[s], 1);
      ptx::mbar_init(&a_empty[s], FOLD ? 5 : 1);          // FOLD: the 4 statistics warps read the tile too
      ptx::mbar_init(&a_ready[s], 4);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&d1_full[s], 1);
      ptx::mbar_init(&d1_empty[s], 8);
      ptx::mbar_init(&h_full[s], 8);
      ptx::mbar_init(&h_empty[s], 1);
    }
    ptx::mbar_init(d2_full, 1);
    ptx::mbar_init(d2_empty, 4);
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int num_tiles = (a.M + Cfg::BM - 1) / Cfg::BM;
  pdl_trigger();                  // TMEM is allocated: dependents may start their prologue where SMs free up
  if (warp != 0) pdl_wait();      // the weight-stream producer touches only weights and may run ahead of the previous kernel

  if (warp == 3) {
    // ===================== y-tile producer ==================================================================
    if (ptx::elect_one()) {
      int it = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
        const int buf = it % Cfg::A_BUFS;
        const uint32_t use = it / Cfg::A_BUFS;
        ptx::mbar_wait(&a_empty[buf], (use & 1) ^ 1);
        uint8_t* sa = smem + Cfg::OFF_A + buf * Cfg::KB1 * Cfg::A_TILE;
        ptx::mbar_arrive_expect_tx(&a_full[buf], Cfg::KB1 * Cfg::A_TILE);
        if (GP) {
          ptx::tma_load_3d(sa, &tmY, &a_full[buf], 0, tile * (Cfg::BM / 32), 0);   // box {32 rows x 16 B, 4, C / 8 groups}
        } else {
          for (int kb = 0; kb < Cfg::KB1; ++kb)
            ptx::tma_load_2d(sa + kb * Cfg::A_TILE, &tmY, &a_full[buf], kb * Cfg::BK, tile * Cfg::BM);
        }
      }
    }
  } else if (warp == 0) {
    // ===================== weight-stream producer ===========================================================
    if (ptx::elect_one()) {
      int slot = 0;
      uint32_t phase = 0;
      auto next_slot = [&]() -> uint8_t* {
        ptx::mbar_wait(&ring_empty[slot], phase ^ 1);
        return smem + Cfg::OFF_RING + slot * Cfg::SLOT;
      };
      auto advance = [&]() {
        if (++slot == Cfg::SLOTS) {
          slot = 0;
          phase ^= 1;
        }
      };
      auto load_w2 = [&](int hh) {
        for (int kb = 0; kb < Cfg::KB2; ++kb) {
          uint8_t* dst = next_slot();
          ptx::mbar_arrive_expect_tx(&ring_full[slot], Cfg::W2_TILE);
          ptx::tma_load_2d(dst, &tmW2, &ring_full[slot], hh * Cfg::NH + kb * Cfg::BK, 0);
          advance();
        }
      };
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        for (int h = 0; h < Cfg::NC; ++h) {
          for (int kb = 0; kb < Cfg::KB1; ++kb) {
            uint8_t* dst = next_slot();
            ptx::mbar_arrive_expect_tx(&ring_full[slot], Cfg::W1_TILE);
            ptx::tma_load_2d(dst, &tmW1, &ring_full[slot], kb * Cfg::BK, h * Cfg::NH);
            advance();
          }
          if (h >= 1) load_w2(h - 1);
        }
        load_w2(Cfg::NC - 1);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer ========================================================================
    if (ptx::elect_one()) {
      constexpr uint32_t idesc1 = ptx::umma_idesc_bf16(Cfg::BM, Cfg::NH);
      constexpr uint32_t idesc2 = ptx::umma_idesc_bf16(Cfg::BM, C);
      const uint32_t d2 = tmem_base + Cfg::D2_COL;
      int slot = 0;
      uint32_t phase = 0;
      auto advance = [&]() {
        if (++slot == Cfg::SLOTS) {
          slot = 0;
          phase ^= 1;
        }
      };
      int it = 0;
      uint32_t gc = 0;                                  // global chunk counter (selects D1 / H buffers and parities)
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
        const int abuf = it % Cfg::A_BUFS;
        const uint32_t ause = it / Cfg::A_BUFS;
        const uint32_t sa = ptx::smem_u32(smem + Cfg::OFF_A + abuf * Cfg::KB1 * Cfg::A_TILE);
        auto gemm2 = [&](int hh, uint32_t gch) {
          const int hb = gch & 1;
          ptx::mbar_wait(&h_full[hb], (gch >> 1) & 1);          // hidden tile written by the epilogue warps
          if (hh == 0) ptx::mbar_wait(d2_empty, (it & 1) ^ 1);  // previous tile's D2 drained
          ptx::tc_fence_after();
          const uint32_t sh = ptx::smem_u32(smem + Cfg::OFF_H + hb * Cfg::KB2 * Cfg::H_TILE);
          for (int kb = 0; kb < Cfg::KB2; ++kb) {
            ptx::mbar_wait(&ring_full[slot], phase);
            ptx::tc_fence_after();
            const uint64_t da = ptx::umma_desc_sw128_kmajor(sh + kb * Cfg::H_TILE);
            const uint64_t db = ptx::umma_desc_sw128_kmajor(ptx::smem_u32(smem + Cfg::OFF_RING + slot * Cfg::SLOT));
#pragma unroll
            for (int k = 0; k < Cfg::BK / 16; ++k)
              ptx::umma_bf16(d2, da + 2 * k, db + 2 * k, idesc2, (hh | kb | k) != 0 ? 1u : 0u);
            ptx::umma_commit(&ring_empty[slot]);
            advance();
          }
          ptx::umma_commit(&h_empty[hb]);
        };
        ptx::mbar_wait((ln && !FOLD) ? &a_ready[abuf] : &a_full[abuf], ause & 1);
        ptx::tc_fence_after();
        for (int h = 0; h < Cfg::NC; ++h, ++gc) {
          const int db1 = gc & 1;
          ptx::mbar_wait(&d1_empty[db1], ((gc >> 1) & 1) ^ 1);
          ptx::tc_fence_after();
          const uint32_t d1 = tmem_base + Cfg::D1_COL + db1 * Cfg::NH;
          for (int kb = 0; kb < Cfg::KB1; ++kb) {
            ptx::mbar_wait(&ring_full[slot], phase);
            ptx::tc_fence_after();
            const uint64_t da = GP ? ptx::umma_desc_nosw_kmajor(sa + kb * Cfg::A_TILE, Cfg::BM * 16, 128)
                                   : ptx::umma_desc_sw128_kmajor(sa + kb * Cfg::A_TILE);
            const uint64_t db = ptx::umma_desc_sw128_kmajor(ptx::smem_u32(smem + Cfg::OFF_RING + slot * Cfg::SLOT));
#pragma unroll
            for (int k = 0; k < Cfg::BK / 16; ++k)
              if (kb * Cfg::BK + k * 16 < C)
                ptx::umma_bf16(d1, da + (GP ? k * (4096 >> 4) : 2 * k), db + 2 * k, idesc1, (kb | k) != 0 ? 1u : 0u);
            ptx::umma_commit(&ring_empty[slot]);
            advance();
          }
          ptx::umma_commit(&d1_full[db1]);
          if (h == Cfg::NC - 1) ptx::umma_commit(&a_empty[abuf]);   // y tile no longer needed
          if (h >= 1) gemm2(h - 1, gc - 1);
        }
        gemm2(Cfg::NC - 1, gc - 1);
        ptx::umma_commit(d2_full);
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ===================== epilogue-1 warps (8): D1 -> +b1 -> GELU -> bf16 -> swizzled hidden tile ==============
    // (two 32-column halves per chunk: keeps the live register set under the 128 registers of a 512-thread CTA)
    const int ew = warp - 4;
    const int quad = warp & 3;
    const int group = ew >> 2;
    const int row_in_tile = quad * 32 + lane;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    uint32_t gc = 0;
    LnFold fold{0ull, 0ull, ptx::smem_u32(sb1), ptx::smem_u32(ss1)};
    int it1 = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it1) {
      for (int h = 0; h < Cfg::NC; ++h, ++gc) {
        const int buf = gc & 1;
        const uint32_t par = (gc >> 1) & 1;
        ptx::mbar_wait(&d1_full[buf], par);
        ptx::tc_fence_after();
        const uint32_t t0 = lane_base + Cfg::D1_COL + buf * Cfg::NH + group * 64;
        const float* bias = sb1 + h * Cfg::NH + group * 64;
        if (FOLD && h == 0) {                           // this tile's row statistics (written by the epilogue-2 warps)
          const int abuf = it1 % Cfg::A_BUFS;
          ptx::mbar_wait(&a_ready[abuf], (it1 / Cfg::A_BUFS) & 1);
          const float2 stt = sstat[(it1 & 1) * Cfg::BM + row_in_tile];
          fold.rstd2 = f2_pack(stt.x, stt.x);
          fold.nmr2 = f2_pack(stt.y, stt.y);
        }
        // this warp group's 64 hidden columns are k-block `group` of the hidden tile: one 128 B swizzled row per lane
        uint8_t* hrow = smem + Cfg::OFF_H + (buf * Cfg::KB2 + group) * Cfg::H_TILE + row_in_tile * 128;
        uint32_t ra[32];
        ptx::tmem_ld_32x32b_x32(t0, ra);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          uint32_t packed[16];
          {
            float2 o[16];
            bias_gelu_tile16_sp<true, FOLD>(ra, bias + 32 * half, o, fold);   // 2 * gelu, see sgamma
#pragma unroll
            for (int j = 0; j < 16; ++j) packed[j] = Pair<bf16>::pack(o[j].x, o[j].y);
          }
          if (half == 0) {
            ptx::tmem_ld_32x32b_x32(t0 + 32, ra);                 // second half's accumulators
            ptx::mbar_wait(&h_empty[buf], par ^ 1);               // GEMM2(h-2) finished reading this hidden buffer
          }
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(hrow + (((4 * half + q) ^ (row_in_tile & 7)) << 4)) =
                make_uint4(packed[4 * q], packed[4 * q + 1], packed[4 * q + 2], packed[4 * q + 3]);
          if (half == 0) {
            ptx::tmem_ld_wait();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&d1_empty[buf]);      // D1 buffer free for GEMM1(h+2)
          }
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&h_full[buf]);
      }
    }
  } else if (warp >= 12) {
    // ===================== epilogue-2 warps (4, one per TMEM lane quadrant), off the critical path ==============
    // D2 -> +b2, *gamma, +residual -> bf16 -> TMA store while the epilogue-1 warps already work on the next tile.
    // Residual chunks arrive by cp.async (coalesced 16 B pieces, zero-filled beyond M) one chunk ahead, into the same
    // 2 KB ping-pong tile that then stages the output chunk.
    constexpr int NCH = C / 32;
    const int quad = warp & 3;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    uint8_t* stg = smem + Cfg::OFF_STG + quad * 4096;
    const int sw64 = (lane >> 1) & 3;
    const int ld_piece = lane & 3, ld_row = lane >> 2;
    // LayerNorm mode: this warp normalises its 32 rows of tile `j` in place as soon as the tile has landed
    auto ln_tile = [&](int j) {
      const int buf = j % Cfg::A_BUFS;
      ptx::mbar_wait(&a_full[buf], (j / Cfg::A_BUFS) & 1);
      const int r = quad * 32 + lane;
      uint8_t* base = smem + Cfg::OFF_A + buf * Cfg::KB1 * Cfg::A_TILE + r * 128;
      if (GP)
        ln_row_in_smem<C>([&](int ch) { return base - r * 128 + ch * (Cfg::BM * 16) + r * 16; }, slnw, slnb);
      else
        ln_row_in_smem<C>([&](int ch) { return base + (ch >> 3) * Cfg::A_TILE + (((ch & 7) ^ (r & 7)) << 4); }, slnw, slnb);
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&a_ready[buf]);
    };
    // FOLD mode: only the row statistics are needed (by the GELU epilogue, not by GEMM1): the tile is read, not rewritten
    auto stats_tile = [&](int j) {
      const int buf = j % Cfg::A_BUFS;
      ptx::mbar_wait(&a_full[buf], (j / Cfg::A_BUFS) & 1);
      const int r = quad * 32 + lane;
      uint8_t* base = smem + Cfg::OFF_A + buf * Cfg::KB1 * Cfg::A_TILE;
      sstat[(j & 1) * Cfg::BM + r] =
          GP ? ln_row_stats_smem<C>([&](int ch) { return base + ch * (Cfg::BM * 16) + r * 16; })
             : ln_row_stats_smem<C>([&](int ch) { return base + r * 128 + (ch >> 3) * Cfg::A_TILE + (((ch & 7) ^ (r & 7)) << 4); });
      __syncwarp();
      if (lane == 0) {
        ptx::mbar_arrive(&a_ready[buf]);
        ptx::mbar_arrive(&a_empty[buf]);
      }
    };
    if (FOLD && (int)blockIdx.x < num_tiles) stats_tile(0);
    if (!FOLD && ln && (int)blockIdx.x < num_tiles) ln_tile(0);
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int row0 = tile * Cfg::BM + quad * 32;
      if (FOLD && tile + (int)gridDim.x < num_tiles) stats_tile(it + 1);
      if (!FOLD && ln && tile + (int)gridDim.x < num_tiles) ln_tile(it + 1);
      auto fetch_resid = [&](int c) {
        uint8_t* dst = stg + (c & 1) * 2048;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int rr = ld_row + 8 * q;
          const int r = row0 + rr;
          const bf16* src = GP ? a.x + ((size_t)(c * 4 + ld_piece) * (((size_t)a.M + 127) / 128 * 128) + (r < a.M ? r : 0)) * 8
                               : a.x + (size_t)(r < a.M ? r : 0) * C + c * 32 + ld_piece * 8;
          const uint32_t d = GP ? ptx::smem_u32(dst + ld_piece * 512 + rr * 16)
                                : ptx::smem_u32(dst + rr * 64 + ((ld_piece ^ ((rr >> 1) & 3)) << 4));
          const int nbytes = r < a.M ? 16 : 0;
          asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(nbytes) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
      };
      if (lane == 0) ptx::tma_store_wait_read<0>();              // previous tile's stores have read both tiles
      __syncwarp();
      fetch_resid(0);
      ptx::mbar_wait(d2_full, it & 1);
      ptx::tc_fence_after();
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        uint8_t* tbuf = stg + (c & 1) * 2048;
        uint32_t r[32];
        ptx::tmem_ld_32x32b_x32(lane_base + Cfg::D2_COL + c * 32, r);
        if (c + 1 < NCH) {
          if (c >= 1) {   // tile (c+1)&1 is the source of chunk c-1's store, the MOST RECENT bulk group: wait for all of
            // them (round 1 waited with <1>, i.e. not for that one -- a write-after-read race that the slower smem reads
            // of the 16-byte-granular 3-D store of the planar layout turned into sporadic corruption)
            if (lane == 0) ptx::tma_store_wait_read<0>();
            __syncwarp();
          }
          fetch_resid(c + 1);
          asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
          asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        ptx::tmem_ld_wait();
        if (c == NCH - 1) {
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(d2_empty);             // D2 free for the next tile's GEMM2
        }
        __syncwarp();
        uint4 res[4];
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4)
          res[j4] = *reinterpret_cast<const uint4*>(GP ? tbuf + j4 * 512 + lane * 16 : tbuf + lane * 64 + ((j4 ^ sw64) << 4));
        __syncwarp();
        const int n = c * 32;
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const int j = j4 * 8;
          const float4 bA = *reinterpret_cast<const float4*>(sb2 + n + j);
          const float4 bB = *reinterpret_cast<const float4*>(sb2 + n + j + 4);
          const float4 gA = *reinterpret_cast<const float4*>(sgamma + n + j);
          const float4 gB = *reinterpret_cast<const float4*>(sgamma + n + j + 4);
          float2 f;
          uint4 o;
          f = Pair<bf16>::unpack(res[j4].x);
          o.x = Pair<bf16>::pack(fmaf(gA.x, __uint_as_float(r[j + 0]), bA.x + f.x), fmaf(gA.y, __uint_as_float(r[j + 1]), bA.y + f.y));
          f = Pair<bf16>::unpack(res[j4].y);
          o.y = Pair<bf16>::pack(fmaf(gA.z, __uint_as_float(r[j + 2]), bA.z + f.x), fmaf(gA.w, __uint_as_float(r[j + 3]), bA.w + f.y));
          f = Pair<bf16>::unpack(res[j4].z);
          o.z = Pair<bf16>::pack(fmaf(gB.x, __uint_as_float(r[j + 4]), bB.x + f.x), fmaf(gB.y, __uint_as_float(r[j + 5]), bB.y + f.y));
          f = Pair<bf16>::unpack(res[j4].w);
          o.w = Pair<bf16>::pack(fmaf(gB.z, __uint_as_float(r[j + 6]), bB.z + f.x), fmaf(gB.w, __uint_as_float(r[j + 7]), bB.w + f.y));
          *reinterpret_cast<uint4*>(GP ? tbuf + j4 * 512 + lane * 16 : tbuf + lane * 64 + ((j4 ^ sw64) << 4)) = o;
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          if (GP) ptx::tma_store_3d(&tmOut, tbuf, 0, row0 >> 5, c * 4);   // box {32 rows x 16 B, 1, 4 groups}
          else ptx::tma_store_2d(&tmOut, tbuf, n, row0);
          ptx::tma_store_commit();
        }
      }
    }
    if (lane == 0) ptx::tma_store_wait_read<0>();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// =====================================================================================================================
// C = 96 (stage 0, the largest M): WEIGHT-RESIDENT variant.  W1 (384 x 96) and W2 (96 x 384) are 144 KB of bf16 -- they
// are TMA-loaded ONCE per persistent CTA and stay in shared memory, so the steady state streams only the y tile in and
// the x tile out.  (The streaming variant above re-read 147 KB of weights from L2 per 128-row tile and, with a ring only
// one hidden chunk deep, exposed one L2 round trip per chunk: 12.7 k cycles per tile against ~2.3 k of MMA work.)
// K = 96 is split 64 + 32: the first 64 columns use 128B-swizzled tiles, the 32-column tail 64B-swizzled tiles, so no
// shared memory is spent on zero padding (W1 48 + 24 KB, W2 72 KB, y tile 16 + 8 KB, hidden buffers 2 x 16 KB).
//
// Schedule (second version, driven by in-kernel clock traces -- commit 17b9d13 -- and an ncu source-level capture):
//   * the 384 hidden columns are six chunks of 64; epilogue-1 group 0 (warps 4-7) takes the even chunks, group 1
//     (warps 8-11) the odd ones, each into its OWN 128 x 64 hidden buffer (one GEMM2 k-block);
//   * TMEM: D2 x 2 (columns 0 and 128: epilogue-2 of tile i overlaps GEMM2 of tile i+1), D1 x 4 (64 columns each,
//     from column 256);
//   * the MMA thread runs one flat loop over all chunks of all its tiles:  G2(g), then G1(g+4)  -- GEMM1 stays four
//     chunks ahead across tile boundaries, GEMM2 is issued as soon as its hidden buffer is full;
//   * the GELU is software-pipelined in 16-column quarters (common.cuh: gelu_stage_ta4 / gelu_stage_c8_twice_bf16).
// =====================================================================================================================
struct Mlp96 {
  static constexpr int C = 96, HD = 384, BM = 128, NH = 64, NC = 6;   // 64-column hidden chunks
  static constexpr int OFF_W1M = 0;                        // 3 x [128 rows x 64 k]  SW128   48 KB
  static constexpr int OFF_W1T = OFF_W1M + 3 * 16384;      // 3 x [128 rows x 32 k]  SW64    24 KB
  static constexpr int OFF_W2 = OFF_W1T + 3 * 8192;        // 6 x [ 96 rows x 64 k]  SW128   72 KB
  static constexpr int OFF_AM = OFF_W2 + 6 * 12288;        // y tile [128 x 64] SW128        16 KB
  static constexpr int OFF_AT = OFF_AM + 16384;            // y tile [128 x 32] SW64          8 KB
  static constexpr int OFF_H = OFF_AT + 8192;              // hidden tile 2 x [128 x 64]     32 KB
  static constexpr int OFF_STG = OFF_H + 32768;            // 8 warps x 2 KB                 16 KB
  static constexpr int OFF_BAR = OFF_STG + 8 * 2048;
  static constexpr int OFF_VEC = OFF_BAR + 256;
  static constexpr int SMEM_BYTES = OFF_VEC + (3 * HD + 4 * C) * 4 + 2 * BM * 8 + 1024;   // + {b1, s} interleaved [2 x 4C], row stats [2][128]
  static constexpr int D2_COL = 0, D2_STRIDE = 128, D1_COL = 256, TMEM_COLS = 512;   // D2 x2 | D1 x4 (64 columns each)
  static constexpr int W_BYTES = 3 * 16384 + 3 * 8192 + 6 * 12288;
  static_assert(SMEM_BYTES <= 227 * 1024, "smem budget");
};

// GP = group-planar activations: y and x are [C/8][M][8] (16-byte channel groups as planes), the layout the tensor-core
// depthwise conv reads and writes with full cache lines; the y tile then arrives as ONE 3-D TMA box {8, 128 rows, 12
// groups} = the un-swizzled canonical K-major operand layout ([group][row][16 B]: K-adjacent core matrices 2 KB apart).
template <bool GP, bool FOLD>
__global__ void __launch_bounds__(512, 1)
    mlp_fused96_kernel(const __grid_constant__ CUtensorMap tmYm, const __grid_constant__ CUtensorMap tmYt,
                       const __grid_constant__ CUtensorMap tmW1m, const __grid_constant__ CUtensorMap tmW1t,
                       const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmOut, MlpArgs a) {
  using Cfg = Mlp96;
  constexpr int C = 96;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* w_full = bars;            // weights landed (once)
  uint64_t* a_full = bars + 1;
  uint64_t* a_empty = bars + 2;
  uint64_t* d1_full = bars + 3;       // [4]  GEMM1 accumulators: ring of four 64-column buffers
  uint64_t* d1_empty = bars + 7;      // [4]
  uint64_t* h_full = bars + 11;       // [2]  hidden tile: one 128 x 64 buffer per epilogue-1 warp group
  uint64_t* h_empty = bars + 13;      // [2]
  uint64_t* d2_full = bars + 15;      // [2]  D2 is double-buffered: epilogue-2 of tile i overlaps GEMM2 of tile i+1
  uint64_t* d2_empty = bars + 17;     // [2]
  uint64_t* a_ready = bars + 19;      // y tile normalised in place (LayerNorm mode only)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 20);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  float* sb1 = reinterpret_cast<float*>(smem + Cfg::OFF_VEC);
  float* sb2 = sb1 + Cfg::HD;
  float* sgamma = sb2 + C;
  float* slnw = sgamma + C;
  float* slnb = slnw + C;
  float* ss1 = slnb + C;                                          // FOLD: {b1[2q], b1[2q+1], s[2q], s[2q+1]} per column pair
  float2* sstat = reinterpret_cast<float2*>(ss1 + 2 * Cfg::HD);   // FOLD: [2][128] (rstd, -mean rstd) per row
  const bool ln = a.ln_w != nullptr;
  for (int i = threadIdx.x; i < Cfg::HD; i += blockDim.x) sb1[i] = a.b1[i];
  if (FOLD)
    for (int i = threadIdx.x; i < Cfg::HD; i += blockDim.x) {
      ss1[4 * (i >> 1) + (i & 1)] = a.b1[i];
      ss1[4 * (i >> 1) + 2 + (i & 1)] = a.ln_s[i];
    }
  if (ln)
    for (int i = threadIdx.x; i < C; i += blockDim.x) {
      slnw[i] = a.ln_w[i];
      slnb[i] = a.ln_b[i];
    }
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    // the hidden tile holds 2 * gelu(.), so  x + gamma (0.5 acc + b2) = x + (0.5 gamma) acc + gamma b2:
    sgamma[i] = 0.5f * a.gamma[i];       // multiplies the GEMM2 accumulator
    sb2[i] = a.gamma[i] * a.b2[i];       // added together with the residual
  }
  if (warp == 0 && ptx::elect_one()) {
    ptx::prefetch_tensormap(&tmYm);
    ptx::prefetch_tensormap(&tmYt);
    ptx::prefetch_tensormap(&tmW1m);
    ptx::prefetch_tensormap(&tmW1t);
    ptx::prefetch_tensormap(&tmW2);
    ptx::prefetch_tensormap(&tmOut);
  }
  if (warp == 1 && ptx::elect_one()) {
    ptx::mbar_init(w_full, 1);
    ptx::mbar_init(a_full, 1);
    ptx::mbar_init(a_empty, FOLD ? 5 : 1);                // FOLD: the 4 statistics warps read the tile too
    ptx::mbar_init(a_ready, 4);
    for (int s = 0; s < 4; ++s) {
      ptx::mbar_init(&d1_full[s], 1);
      ptx::mbar_init(&d1_empty[s], 4);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&h_full[s], 4);
      ptx::mbar_init(&h_empty[s], 1);
      ptx::mbar_init(&d2_full[s], 1);
      ptx::mbar_init(&d2_empty[s], 4);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int num_tiles = (a.M + Cfg::BM - 1) / Cfg::BM;
  pdl_trigger();                  // TMEM is allocated: dependents may start their prologue where SMs free up
  if (warp != 0) pdl_wait();      // warp 0 first requests the resident weights (144 KB, independent of the previous kernel)

  if (warp == 0) {
    // ===================== producer: weights once, then one y tile per row tile ==============================
    if (ptx::elect_one()) {
      ptx::mbar_arrive_expect_tx(w_full, Cfg::W_BYTES);
      for (int h = 0; h < 3; ++h) {
        ptx::tma_load_2d(smem + Cfg::OFF_W1M + h * 16384, &tmW1m, w_full, 0, h * 128);
        ptx::tma_load_2d(smem + Cfg::OFF_W1T + h * 8192, &tmW1t, w_full, 64, h * 128);
      }
      for (int kb = 0; kb < 6; ++kb) ptx::tma_load_2d(smem + Cfg::OFF_W2 + kb * 12288, &tmW2, w_full, kb * 64, 0);
      pdl_wait();                 // the y tiles are the previous kernel's output
      int it = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
        ptx::mbar_wait(a_empty, (it & 1) ^ 1);
        ptx::mbar_arrive_expect_tx(a_full, 16384 + 8192);
        const int next = tile + gridDim.x;                        // the single y buffer cannot be loaded ahead, but
        if (GP) {                                                 // its HBM latency can: pull the next tile into L2
          ptx::tma_load_3d(smem + Cfg::OFF_AM, &tmYm, a_full, 0, tile * (Cfg::BM / 32), 0);
          if (next < num_tiles) ptx::tma_prefetch_3d(&tmYm, 0, next * (Cfg::BM / 32), 0);
        } else {
          ptx::tma_load_2d(smem + Cfg::OFF_AM, &tmYm, a_full, 0, tile * Cfg::BM);
          ptx::tma_load_2d(smem + Cfg::OFF_AT, &tmYt, a_full, 64, tile * Cfg::BM);
          if (next < num_tiles) {
            ptx::tma_prefetch_2d(&tmYm, 0, next * Cfg::BM);
            ptx::tma_prefetch_2d(&tmYt, 64, next * Cfg::BM);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer ========================================================================
    if (ptx::elect_one()) {
      constexpr uint32_t idesc1 = ptx::umma_idesc_bf16(Cfg::BM, Cfg::NH);
      constexpr uint32_t idesc2 = ptx::umma_idesc_bf16(Cfg::BM, C);
      const uint32_t sbase = ptx::smem_u32(smem);
      const uint64_t dAm = ptx::umma_desc_sw128_kmajor(sbase + Cfg::OFF_AM);
      const uint64_t dAt = ptx::umma_desc_sw64_kmajor(sbase + Cfg::OFF_AT);
      const uint64_t dAg = ptx::umma_desc_nosw_kmajor(sbase + Cfg::OFF_AM, 128 * 16, 128);   // GP: [group][row][16 B]
      ptx::mbar_wait(w_full, 0);
      ptx::tc_fence_after();
      // FLAT schedule over the CTA's hidden chunks g = 6 * tile_iteration + h (64 hidden columns each):
      //   G1(0) .. G1(3) | G2(g), G1(g+4) | ...
      // GEMM1 runs four chunks ahead of GEMM2 through a ring of four TMEM buffers, ACROSS tile boundaries: the two
      // epilogue-1 warp groups work on chunks g and g+1 at the same time (even / odd chunks), each filling its OWN
      // hidden-tile buffer, so neither the epilogue nor this thread ever waits for the other within a chunk.  (History,
      // from clock traces: per-tile order with one 128-column hidden buffer -> epilogue idle 1.5 k of 8.9 k cycles per
      // tile at tile boundaries and ~0.6 k per chunk waiting for GEMM2 to release the buffer.)
      const int my_tiles = (int)blockIdx.x < num_tiles ? (num_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
      const uint32_t total = (uint32_t)Cfg::NC * my_tiles;
      auto gemm1 = [&](uint32_t g, int h, int it) {
        if (h == 0) {
          ptx::mbar_wait((ln && !FOLD) ? a_ready : a_full, it & 1);
          ptx::tc_fence_after();
        }
        const int db1 = g & 3;
        ptx::mbar_wait(&d1_empty[db1], ((g >> 2) & 1) ^ 1);
        ptx::tc_fence_after();
        const uint32_t d1 = tmem_base + Cfg::D1_COL + db1 * Cfg::NH;
        // W1 rows [64 h, 64 h + 64): second half of a 128-row tile starts 64 rows = 8 swizzle atoms further
        const uint64_t dBm = ptx::umma_desc_sw128_kmajor(sbase + Cfg::OFF_W1M + (h >> 1) * 16384 + (h & 1) * 8192);
        const uint64_t dBt = ptx::umma_desc_sw64_kmajor(sbase + Cfg::OFF_W1T + (h >> 1) * 8192 + (h & 1) * 4096);
        if (GP) {   // k-step ks covers channel groups 2 ks, 2 ks + 1: 2 x 2 KB further per step
#pragma unroll
          for (int k = 0; k < 4; ++k) ptx::umma_bf16(d1, dAg + k * (4096 >> 4), dBm + 2 * k, idesc1, k != 0 ? 1u : 0u);
#pragma unroll
          for (int k = 0; k < 2; ++k) ptx::umma_bf16(d1, dAg + (4 + k) * (4096 >> 4), dBt + 2 * k, idesc1, 1u);
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k) ptx::umma_bf16(d1, dAm + 2 * k, dBm + 2 * k, idesc1, k != 0 ? 1u : 0u);
#pragma unroll
          for (int k = 0; k < 2; ++k) ptx::umma_bf16(d1, dAt + 2 * k, dBt + 2 * k, idesc1, 1u);
        }
        ptx::umma_commit(&d1_full[db1]);
        if (h == Cfg::NC - 1) ptx::umma_commit(a_empty);          // y tile consumed: the producer may load the next
      };
      auto gemm2 = [&](uint32_t g, int h, int it) {
        const int hb = g & 1;
        ptx::mbar_wait(&h_full[hb], (g >> 1) & 1);
        if (h == 0) ptx::mbar_wait(&d2_empty[it & 1], ((it >> 1) & 1) ^ 1);
        ptx::tc_fence_after();
        const uint32_t d2 = tmem_base + Cfg::D2_COL + (it & 1) * Cfg::D2_STRIDE;
        const uint64_t da = ptx::umma_desc_sw128_kmajor(sbase + Cfg::OFF_H + hb * 16384);
        const uint64_t db = ptx::umma_desc_sw128_kmajor(sbase + Cfg::OFF_W2 + h * 12288);
#pragma unroll
        for (int k = 0; k < 4; ++k) ptx::umma_bf16(d2, da + 2 * k, db + 2 * k, idesc2, (h | k) != 0 ? 1u : 0u);
        ptx::umma_commit(&h_empty[hb]);
        if (h == Cfg::NC - 1) ptx::umma_commit(&d2_full[it & 1]);
      };
      // GEMM1 look-ahead = ring depth: chunk g+4 reuses chunk g's buffer, which the epilogue released half-way
      // through chunk g, i.e. before the h_full(g) that gemm2(g) has just waited for
      constexpr int LA = 4;
      int h1 = 0, it1 = 0;                     // chunk / tile iteration of the next GEMM1
      uint32_t g1 = 0;
      auto issue_gemm1 = [&]() {
        if (g1 < total) {
          gemm1(g1, h1, it1);
          ++g1;
          if (++h1 == Cfg::NC) {
            h1 = 0;
            ++it1;
          }
        }
      };
      for (int i = 0; i < LA; ++i) issue_gemm1();
      int h = 0, it = 0;
      for (uint32_t g = 0; g < total; ++g) {
        gemm2(g, h, it);        // first: the epilogue group that filled this hidden buffer waits for its release
        issue_gemm1();          // then top up the GEMM1 ring (four chunks ahead, never urgent)
        if (++h == Cfg::NC) {
          h = 0;
          ++it;
        }
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ===================== epilogue-1 warps (2 groups x 4): D1 -> +b1 -> GELU -> bf16 -> swizzled hidden tile =====
    // Group 0 (warps 4-7) takes the even 64-column chunks, group 1 (warps 8-11) the odd ones; a warp owns 32 rows x
    // 64 hidden columns of its chunk.  The two warps that share a scheduler therefore sit in different chunks, out of
    // phase, and each group writes its own 16 KB hidden buffer.
    const int ew = warp - 4;
    const int quad = warp & 3;
    const int group = ew >> 2;
    const int row_in_tile = quad * 32 + lane;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    LnFold fold{0ull, 0ull, ptx::smem_u32(sb1), ptx::smem_u32(ss1)};
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      if (FOLD) {                                       // this tile's row statistics (written by the epilogue-2 warps)
        ptx::mbar_wait(a_ready, it & 1);
        const float2 stt = sstat[(it & 1) * Cfg::BM + row_in_tile];
        fold.rstd2 = f2_pack(stt.x, stt.x);
        fold.nmr2 = f2_pack(stt.y, stt.y);
      }
      for (int hc = 0; hc < Cfg::NC / 2; ++hc) {
        const int h = 2 * hc + group;
        const uint32_t gc = (uint32_t)Cfg::NC * it + h;
        const int buf = gc & 3;
        ptx::mbar_wait(&d1_full[buf], (gc >> 2) & 1);
        ptx::tc_fence_after();
        const uint32_t t0 = lane_base + Cfg::D1_COL + buf * Cfg::NH;
        const uint32_t bias = ptx::smem_u32(sb1 + h * Cfg::NH);
        const uint32_t hrow = ptx::smem_u32(smem + Cfg::OFF_H + group * 16384 + row_in_tile * 128);
        // Four 16-column quarters, software-pipelined:  A(0) | T(0)+A(1) | C(0) | T(1)+A(2) | C(1) | T(2)+A(3) | ...
        // (A = bias, polynomial: FMA pipe; T = 2 x MUFU.TANH per pair: XU pipe; C = x + x t, pack, store: FMA pipe).
        uint32_t raA[16], raB[16];
        GeluPair gA[8], gB[8];
        uint32_t pk[8] = {};
        auto store_quarter = [&](int qi) {
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(hrow + (((2 * qi) ^ (row_in_tile & 7)) << 4)),
                       "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3])
                       : "memory");
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(hrow + (((2 * qi + 1) ^ (row_in_tile & 7)) << 4)),
                       "r"(pk[4]), "r"(pk[5]), "r"(pk[6]), "r"(pk[7])
                       : "memory");
        };
        ptx::tmem_ld_32x32b_x16(t0, raA);
        ptx::tmem_ld_32x32b_x16(t0 + 16, raB);
        ptx::tmem_ld_wait_dep(raA, raB);
        gelu_stage_ta4<false, true, FOLD>(nullptr, gA, raA, bias, fold);                       // A(0)
        gelu_stage_ta4<false, true, FOLD>(nullptr, gA + 4, raA + 8, bias + 32, fold);
        ptx::tmem_ld_32x32b_x16(t0 + 32, raA);
        gelu_stage_ta4<true, true, FOLD>(gA, gB, raB, bias + 64, fold);                        // T(0) + A(1)
        gelu_stage_ta4<true, true, FOLD>(gA + 4, gB + 4, raB + 8, bias + 96, fold);
        ptx::tmem_ld_32x32b_x16(t0 + 48, raB);
        gelu_stage_c8_twice_bf16(gA, pk);                                          // C(0)
        ptx::mbar_wait(&h_empty[group], ((gc >> 1) & 1) ^ 1);     // GEMM2 of this group's previous chunk has read the buffer
        store_quarter(0);
        ptx::tmem_ld_wait_dep(raA, raB);
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&d1_empty[buf]);          // all of this warp's D1 reads landed: free for GEMM1(g+4)
        gelu_stage_ta4<true, true, FOLD>(gB, gA, raA, bias + 128, fold);                       // T(1) + A(2)
        gelu_stage_ta4<true, true, FOLD>(gB + 4, gA + 4, raA + 8, bias + 160, fold);
        gelu_stage_c8_twice_bf16(gB, pk);                                          // C(1)
        store_quarter(1);
        gelu_stage_ta4<true, true, FOLD>(gA, gB, raB, bias + 192, fold);                       // T(2) + A(3)
        gelu_stage_ta4<true, true, FOLD>(gA + 4, gB + 4, raB + 8, bias + 224, fold);
        gelu_stage_c8_twice_bf16(gA, pk);                                          // C(2)
        store_quarter(2);
        gelu_stage_ta4<true, false>(gB, nullptr, nullptr, 0);                      // T(3)
        gelu_stage_ta4<true, false>(gB + 4, nullptr, nullptr, 0);
        gelu_stage_c8_twice_bf16(gB, pk);                                          // C(3)
        store_quarter(3);
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&h_full[group]);
      }
    }
  } else if (warp >= 12) {
    // ===================== epilogue-2 warps (4, one per TMEM lane quadrant) =====================================
    // D2 -> +b2, *gamma, +residual -> bf16 -> TMA store, OFF the critical path: while these warps finish tile i the
    // epilogue-1 warps are already producing the hidden tiles of tile i+1 (a clock trace showed epilogue-2, a chain of
    // dependent latencies -- residual fetch, smem transposes, TMEM loads -- taking 3.3 k of the 11 k cycles per tile
    // when the same 8 warps did both).  The residual chunk is brought in with cp.async (coalesced 16 B pieces,
    // zero-filled beyond M) one chunk ahead, into the same 2 KB ping-pong tile that later stages the output.
    const int quad = warp & 3;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    uint8_t* stg = smem + Cfg::OFF_STG + quad * 4096;            // 2 x 2 KB ping-pong tiles
    const int sw64 = (lane >> 1) & 3;
    const int ld_piece = lane & 3, ld_row = lane >> 2;
    // LayerNorm mode: this warp normalises its 32 rows of tile `j` in place as soon as the tile has landed (columns
    // 0..63 in the 128B-swizzled tile, 64..95 in the 64B-swizzled tail tile)
    auto ln_tile = [&](int j) {
      ptx::mbar_wait(a_full, j & 1);
      const int r = quad * 32 + lane;
      uint8_t* am = smem + Cfg::OFF_AM + r * 128;
      uint8_t* at = smem + Cfg::OFF_AT + r * 64;
      if (GP)
        ln_row_in_smem<C>([&](int ch) { return smem + Cfg::OFF_AM + ch * 2048 + r * 16; }, slnw, slnb);
      else
        ln_row_in_smem<C>([&](int ch) { return ch < 8 ? am + ((ch ^ (r & 7)) << 4) : at + (((ch - 8) ^ ((r >> 1) & 3)) << 4); },
                          slnw, slnb);
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(a_ready);
    };
    // FOLD mode: only the row statistics are needed (by the GELU epilogue, not by GEMM1): the tile is read, not rewritten
    auto stats_tile = [&](int j) {
      ptx::mbar_wait(a_full, j & 1);
      const int r = quad * 32 + lane;
      uint8_t* am = smem + Cfg::OFF_AM + r * 128;
      uint8_t* at = smem + Cfg::OFF_AT + r * 64;
      sstat[(j & 1) * Cfg::BM + r] =
          GP ? ln_row_stats_smem<C>([&](int ch) { return smem + Cfg::OFF_AM + ch * 2048 + r * 16; })
             : ln_row_stats_smem<C>([&](int ch) { return ch < 8 ? am + ((ch ^ (r & 7)) << 4) : at + (((ch - 8) ^ ((r >> 1) & 3)) << 4); });
      __syncwarp();
      if (lane == 0) {
        ptx::mbar_arrive(a_ready);
        ptx::mbar_arrive(a_empty);
      }
    };
    if (FOLD && (int)blockIdx.x < num_tiles) stats_tile(0);
    if (!FOLD && ln && (int)blockIdx.x < num_tiles) ln_tile(0);
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int row0 = tile * Cfg::BM + quad * 32;
      if (FOLD && tile + (int)gridDim.x < num_tiles) stats_tile(it + 1);
      if (!FOLD && ln && tile + (int)gridDim.x < num_tiles) ln_tile(it + 1);
      auto fetch_resid = [&](int c) {                            // 32 rows x 64 B of chunk c -> tile (c & 1)
        uint8_t* dst = stg + (c & 1) * 2048;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int rr = ld_row + 8 * q;
          const int r = row0 + rr;
          const bf16* src = GP ? a.x + ((size_t)(c * 4 + ld_piece) * (((size_t)a.M + 127) / 128 * 128) + (r < a.M ? r : 0)) * 8
                               : a.x + (size_t)(r < a.M ? r : 0) * C + c * 32 + ld_piece * 8;
          const uint32_t d = GP ? ptx::smem_u32(dst + ld_piece * 512 + rr * 16)
                                : ptx::smem_u32(dst + rr * 64 + ((ld_piece ^ ((rr >> 1) & 3)) << 4));
          const int nbytes = r < a.M ? 16 : 0;
          asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(nbytes) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
      };
      if (lane == 0) ptx::tma_store_wait_read<0>();              // previous tile's stores have read both tiles
      __syncwarp();
      fetch_resid(0);
      ptx::mbar_wait(&d2_full[it & 1], (it >> 1) & 1);
      ptx::tc_fence_after();
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        uint8_t* tbuf = stg + (c & 1) * 2048;
        uint32_t r[32];
        ptx::tmem_ld_32x32b_x32(lane_base + Cfg::D2_COL + (it & 1) * Cfg::D2_STRIDE + c * 32, r);
        if (c + 1 < 3) {
          if (c >= 1) {   // tile (c+1)&1 is the source of chunk c-1's store, the MOST RECENT bulk group: wait for all of
            // them (round 1 waited with <1>, i.e. not for that one -- a write-after-read race that the slower smem reads
            // of the 16-byte-granular 3-D store of the planar layout turned into sporadic corruption)
            if (lane == 0) ptx::tma_store_wait_read<0>();
            __syncwarp();
          }
          fetch_resid(c + 1);
          asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
          asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        ptx::tmem_ld_wait();
        if (c == 2) {
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&d2_empty[it & 1]);   // this D2 buffer is free for tile i+2's GEMM2
        }
        __syncwarp();
        uint4 res[4];
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4)
          res[j4] = *reinterpret_cast<const uint4*>(GP ? tbuf + j4 * 512 + lane * 16 : tbuf + lane * 64 + ((j4 ^ sw64) << 4));
        __syncwarp();
        const int n = c * 32;
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const int j = j4 * 8;
          const float4 bA = *reinterpret_cast<const float4*>(sb2 + n + j);
          const float4 bB = *reinterpret_cast<const float4*>(sb2 + n + j + 4);
          const float4 gA = *reinterpret_cast<const float4*>(sgamma + n + j);
          const float4 gB = *reinterpret_cast<const float4*>(sgamma + n + j + 4);
          float2 f;
          uint4 o;
          f = Pair<bf16>::unpack(res[j4].x);
          o.x = Pair<bf16>::pack(fmaf(gA.x, __uint_as_float(r[j + 0]), bA.x + f.x), fmaf(gA.y, __uint_as_float(r[j + 1]), bA.y + f.y));
          f = Pair<bf16>::unpack(res[j4].y);
          o.y = Pair<bf16>::pack(fmaf(gA.z, __uint_as_float(r[j + 2]), bA.z + f.x), fmaf(gA.w, __uint_as_float(r[j + 3]), bA.w + f.y));
          f = Pair<bf16>::unpack(res[j4].z);
          o.z = Pair<bf16>::pack(fmaf(gB.x, __uint_as_float(r[j + 4]), bB.x + f.x), fmaf(gB.y, __uint_as_float(r[j + 5]), bB.y + f.y));
          f = Pair<bf16>::unpack(res[j4].w);
          o.w = Pair<bf16>::pack(fmaf(gB.z, __uint_as_float(r[j + 6]), bB.z + f.x), fmaf(gB.w, __uint_as_float(r[j + 7]), bB.w + f.y));
          *reinterpret_cast<uint4*>(GP ? tbuf + j4 * 512 + lane * 16 : tbuf + lane * 64 + ((j4 ^ sw64) << 4)) = o;
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          if (GP) ptx::tma_store_3d(&tmOut, tbuf, 0, row0 >> 5, c * 4);   // box {32 rows x 16 B, 1, 4 groups}
          else ptx::tma_store_2d(&tmOut, tbuf, n, row0);
          ptx::tma_store_commit();
        }
      }
    }
    if (lane == 0) ptx::tma_store_wait_read<0>();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

static int launch_mlp96_resident(const void* y, void* x, const void* w1, const float* b1, const void* w2,
                                 const float* b2, const float* gamma, int M, const float* ln_w, const float* ln_b,
                                 const float* ln_s, bool gp, cudaStream_t st) {
  using Cfg = Mlp96;
  CUtensorMap tmYm, tmYt, tmW1m, tmW1t, tmW2, tmOut;
  int rc;
  if (gp) {
    rc = make_tmap_gp_bf16(&tmYm, y, (uint64_t)M, 12, 128, 12);
    tmYt = tmYm;
  } else {
    rc = make_tmap_2d_bf16(&tmYm, y, 96, (uint64_t)M, 192, 64, 128);
    if (rc != ACX_OK) return rc;
    rc = make_tmap_2d_bf16(&tmYt, y, 96, (uint64_t)M, 192, 32, 128, CU_TENSOR_MAP_SWIZZLE_64B);
  }
  if (rc != ACX_OK) return rc;
  rc = make_tmap_2d_bf16(&tmW1m, w1, 96, 384, 192, 64, 128);
  if (rc != ACX_OK) return rc;
  rc = make_tmap_2d_bf16(&tmW1t, w1, 96, 384, 192, 32, 128, CU_TENSOR_MAP_SWIZZLE_64B);
  if (rc != ACX_OK) return rc;
  rc = make_tmap_2d_bf16(&tmW2, w2, 384, 96, 768, 64, 96);
  if (rc != ACX_OK) return rc;
  rc = gp ? make_tmap_gp_bf16(&tmOut, x, (uint64_t)M, 12, 32, 4)
          : make_tmap_2d_bf16(&tmOut, x, 96, (uint64_t)M, 192, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B);
  if (rc != ACX_OK) return rc;
  ACX_SET_MAX_SMEM((mlp_fused96_kernel<false, false>), Cfg::SMEM_BYTES);
  ACX_SET_MAX_SMEM((mlp_fused96_kernel<true, false>), Cfg::SMEM_BYTES);
  ACX_SET_MAX_SMEM((mlp_fused96_kernel<true, true>), Cfg::SMEM_BYTES);
  int dev = 0, sms = 0;
  ACX_CUDA(cudaGetDevice(&dev));
  ACX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int tiles = ceil_div(M, Cfg::BM);
  MlpArgs a;
  a.x = reinterpret_cast<bf16*>(x);
  a.b1 = b1;
  a.b2 = b2;
  a.gamma = gamma;
  a.M = M;
  a.ln_w = ln_w;
  a.ln_b = ln_b;
  a.ln_s = ln_s;
  const int grid = tiles < sms ? tiles : sms;
  auto kern = gp && ln_s ? mlp_fused96_kernel<true, true> : gp ? mlp_fused96_kernel<true, false> : mlp_fused96_kernel<false, false>;
  ACX_CUDA(launch_pdl(kern, dim3(grid), dim3(512), Cfg::SMEM_BYTES, st, 1, PDL_MLP, tmYm, tmYt, tmW1m, tmW1t, tmW2, tmOut, a));
  return ACX_OK;
}

template <int C>
static int launch_mlp(const void* y, void* x, const void* w1, const float* b1, const void* w2, const float* b2,
                      const float* gamma, int M, const float* ln_w, const float* ln_b, const float* ln_s, bool gp,
                      cudaStream_t st) {
  using Cfg = MlpCfg<C>;
  CUtensorMap tmY, tmW1, tmW2, tmOut;
  ACX_CHECK(!gp || C % 64 == 0, ACX_ERR_UNSUPPORTED, "mlp_fused: the streaming kernel takes group-planar tiles for C %% 64 == 0 only");
  int rc = gp ? make_tmap_gp_bf16(&tmY, y, (uint64_t)M, C / 8, 128, C / 8)
              : make_tmap_2d_bf16(&tmY, y, C, (uint64_t)M, (uint64_t)C * 2, 64, 128);
  if (rc != ACX_OK) return rc;
  rc = make_tmap_2d_bf16(&tmW1, w1, C, Cfg::HD, (uint64_t)C * 2, 64, Cfg::NH);
  if (rc != ACX_OK) return rc;
  rc = make_tmap_2d_bf16(&tmW2, w2, Cfg::HD, C, (uint64_t)Cfg::HD * 2, 64, C);
  if (rc != ACX_OK) return rc;
  rc = gp ? make_tmap_gp_bf16(&tmOut, x, (uint64_t)M, C / 8, 32, 4)
          : make_tmap_2d_bf16(&tmOut, x, C, (uint64_t)M, (uint64_t)C * 2, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B);
  if (rc != ACX_OK) return rc;
  ACX_SET_MAX_SMEM((mlp_fused_kernel<C, false, false>), Cfg::SMEM_BYTES);
  ACX_SET_MAX_SMEM((mlp_fused_kernel<C, true, false>), Cfg::SMEM_BYTES);
  ACX_SET_MAX_SMEM((mlp_fused_kernel<C, true, true>), Cfg::SMEM_BYTES);
  int dev = 0, sms = 0;
  ACX_CUDA(cudaGetDevice(&dev));
  ACX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int tiles = ceil_div(M, Cfg::BM);
  MlpArgs a;
  a.x = reinterpret_cast<bf16*>(x);
  a.b1 = b1;
  a.b2 = b2;
  a.gamma = gamma;
  a.M = M;
  a.ln_w = ln_w;
  a.ln_b = ln_b;
  a.ln_s = ln_s;
  const int grid = tiles < sms ? tiles : sms;
  auto kern = gp && ln_s ? mlp_fused_kernel<C, true, true> : gp ? mlp_fused_kernel<C, true, false> : mlp_fused_kernel<C, false, false>;
  ACX_CUDA(launch_pdl(kern, dim3(grid), dim3(Cfg::THREADS), Cfg::SMEM_BYTES, st, 1, PDL_MLP, tmY, tmW1, tmW2, tmOut, a));
  return ACX_OK;
}

}  // namespace acx

using namespace acx;

static int mlp_fused_dispatch(const char* who, const void* y, void* x, const void* w1, const float* b1, const void* w2,
                              const float* b2, const float* gamma, int M, int C, const float* ln_w, const float* ln_b,
                              const float* ln_s, bool gp, void* stream) {
  ACX_CHECK(!ln_s || (gp && !ln_w && !ln_b), ACX_ERR_ARG,
            "%s: the folded LayerNorm (ln_s) is a group-planar mode and excludes ln_w / ln_b (they are folded into w1 / b1)", who);
  ACX_CHECK(y && x && w1 && b1 && w2 && b2 && gamma, ACX_ERR_ARG, "%s: null pointer", who);
  ACX_CHECK(M > 0, ACX_ERR_ARG, "%s: M must be positive", who);
  ACX_CHECK(((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w1) |
              reinterpret_cast<uintptr_t>(w2)) & 15) == 0,
            ACX_ERR_ARG, "%s: y, x, w1 and w2 must be 16-byte aligned", who);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  switch (C) {
    case 96: return launch_mlp96_resident(y, x, w1, b1, w2, b2, gamma, M, ln_w, ln_b, ln_s, gp, st);
    case 192: return launch_mlp<192>(y, x, w1, b1, w2, b2, gamma, M, ln_w, ln_b, ln_s, gp, st);
    default:
      set_error("%s: C=%d not supported (the fused kernel covers stages 0-1: C = 96, 192; wider stages exceed "
                "the 512 TMEM columns and use acx_gemm_bf16 twice)", who, C);
      return ACX_ERR_UNSUPPORTED;
  }
}

extern "C" int acx_mlp_fused(const void* y, void* x, const void* w1, const float* b1, const void* w2, const float* b2,
                             const float* gamma, int M, int C, void* stream) {
  return mlp_fused_dispatch("mlp_fused", y, x, w1, b1, w2, b2, gamma, M, C, nullptr, nullptr, nullptr, false, stream);
}

// Same, with the Block's channels-last LayerNorm (convnext.py:78) applied to the operand tile on the SM: v is the RAW
// depthwise-conv output (acx_dwconv_tc), never normalised in HBM.
extern "C" int acx_mlp_fused_ln(const void* v, void* x, const float* ln_w, const float* ln_b, const void* w1,
                                const float* b1, const void* w2, const float* b2, const float* gamma, int M, int C,
                                void* stream) {
  ACX_CHECK(ln_w && ln_b, ACX_ERR_ARG, "mlp_fused_ln: null LayerNorm vectors");
  return mlp_fused_dispatch("mlp_fused_ln", v, x, w1, b1, w2, b2, gamma, M, C, ln_w, ln_b, nullptr, false, stream);
}

// Group-planar variant: v and x are [C/8][M][8] bf16 (the 16-byte channel groups of all M rows as planes) -- the layout
// acx_dwconv_tc_gp reads and writes with full cache lines.  ln_w / ln_b may be null (v already normalised).
extern "C" int acx_mlp_fused_gp(const void* v, void* x, const float* ln_w, const float* ln_b, const float* ln_s,
                                const void* w1, const float* b1, const void* w2, const float* b2, const float* gamma,
                                int M, int C, void* stream) {
  ACX_CHECK((ln_w == nullptr) == (ln_b == nullptr), ACX_ERR_ARG, "mlp_fused_gp: ln_w and ln_b must both be given or both be null");
  return mlp_fused_dispatch("mlp_fused_gp", v, x, w1, b1, w2, b2, gamma, M, C, ln_w, ln_b, ln_s, true, stream);
}
