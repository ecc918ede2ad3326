// tcgen05 GEMM:  out[M,N] (bf16) = epi( A[M,K] (bf16) . W[N,K]^T (bf16) ), fp32 accumulation in TMEM.
//
// Persistent, warp-specialised, one CTA per SM:
//   warp 0      TMA producer   (cp.async.bulk.tensor, 128B-swizzled 128x64 / BNx64 tiles)
//   warp 1      MMA issuer     (one elected thread, tcgen05.mma.cta_group::1.kind::f16, M=128, N=BN, K=16)
//   warp 2      TMEM allocator
//   warps 4..   epilogue       (tcgen05.ld 32x32b -> bias / GELU / layer-scale+residual -> bf16 -> global)
// Pipelines: smem ring (full/empty mbarriers, STAGES deep) between TMA and MMA; two TMEM accumulators
// (tmem_full/tmem_empty) between MMA and epilogue, so tile i's epilogue overlaps tile i+1's MMAs.
//
// Used for pwconv1+GELU / pwconv2+gamma+residual (reference convnext.py:79-86) and the 2x2/s2 downsample
// convolutions as GEMMs over the patch matrix (convnext.py:231-234).
#include <stdlib.h>

#include "common.cuh"
#include "ptx.cuh"
#include "tmap.cuh"

namespace acx {

struct GemmArgs {
  bf16* out;
  const float* bias;
  const float* gamma;
  const bf16* resid;
  int M, N, K;
  int out_gp;   // 1: `out` (and `resid`) are group-planar [N/8][Mp][8] (the hand-off layout of the tensor-core depthwise conv)
  int a_gp;     // 1: A is group-planar [K/8][Mp][8]: operand tiles arrive as 3-D boxes in the un-swizzled K-major layout
  const float2* stats;   // EPI_BIAS_GELU_FOLD: per-row (rstd, -mean * rstd) of A (acx_gp_row_stats)
  const float* ln_s;     // EPI_BIAS_GELU_FOLD: s[j] = sum_k W[j, k] of the LayerNorm-folded weights
  int reverse;           // walk the tiles from the last row block to the first: a consumer of a tensor LARGER than L2 that the
                         // previous kernel wrote front to back (pwconv2 reading the 173 MB hidden tensor of stage 2) then
                         // starts with the part that is still in L2 instead of evicting it on the way there
};
constexpr int ACX_EPI_BIAS_GELU_FOLD = 3;   // internal: GELU epilogue with the LayerNorm applied as a rank-1 correction

// CG = 1: one CTA per 128 x BN tile.  CG = 2: a CTA PAIR (cluster of 2, tcgen05 cta_group::2) per 256 x BN tile -- each
// CTA stages its own 128 A rows and HALF of the B rows, so operand traffic from L2 per FLOP drops by a third and the
// smaller stage allows a deeper ring.  The stage-2/3 GEMMs were L2-bandwidth-bound with CG = 1 (ncu: tensor pipe 50 %,
// ~10 TB/s of operand re-reads).
template <int BN_, int NEPI_, int CG_ = 1>
struct GemmCfg {
  static constexpr int BM = 128, BN = BN_, BK = 64, NEPI = NEPI_, CG = CG_;
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = (BN / CG) * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES_RAW = (160 * 1024) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 6 ? 6 : STAGES_RAW;
  static_assert(CG == 1 || BN % 32 == 0, "B halves");
  static constexpr int ACC_STRIDE = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
  static constexpr int TMEM_COLS = 2 * ACC_STRIDE;
  // epilogue: 8 warps = 4 TMEM lane quadrants x 2 column groups; columns are handed out in chunks of 32
  static constexpr int CHUNK = 32;
  static constexpr int NCHUNKS = BN / CHUNK;
  static constexpr int CH_G0 = (NCHUNKS + 1) / 2;      // chunks of column group 0 (group 1 gets the rest)
  static constexpr int THREADS = 128 + 32 * NEPI;
  // per epilogue warp: 2 output staging tiles + 1 residual tile, each 32 rows x 64 B (SWIZZLE_64B)
  static constexpr int STG_TILE = 32 * CHUNK * 2;
  static constexpr int STG_PER_WARP = 3 * STG_TILE;
  static constexpr int OFF_STG = STAGES * STAGE_BYTES;
  static constexpr int OFF_BAR = OFF_STG + NEPI * STG_PER_WARP;
  static constexpr int OFF_VEC = OFF_BAR + 256;        // bias[N] (+ gamma[N]) staged once per CTA (dynamic size)
  static constexpr int VEC_BYTES = 16 * 1024;          // bias up to 3072 columns, gamma up to 1024
  static constexpr int SMEM_BYTES = OFF_VEC + VEC_BYTES + 1024 /*align*/;
  static_assert(NEPI == 8, "epilogue layout assumes 8 warps");
  static_assert(BN % 32 == 0 && BN >= 32 && BN <= 256, "UMMA N constraint for M=128 / 32-column epilogue chunks");
  static_assert(B_BYTES % 1024 == 0, "stage buffers must stay 1024B aligned for SWIZZLE_128B");
  static_assert(SMEM_BYTES <= 227 * 1024, "smem budget");
};

template <int BN, int EPI, int NEPI, int CG>
__global__ void __launch_bounds__(GemmCfg<BN, NEPI, CG>::THREADS, 1)
    umma_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                     const __grid_constant__ CUtensorMap tmOut, GemmArgs g) {
  using Cfg = GemmCfg<BN, NEPI, CG>;
  const uint32_t cta_rank = CG == 2 ? ptx::cluster_ctarank() : 0u;   // 0 = leader of the pair
  const int unit = CG == 2 ? blockIdx.x >> 1 : blockIdx.x;           // persistent work unit (CTA or CTA pair)
  const int num_units = CG == 2 ? gridDim.x >> 1 : gridDim.x;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* empty_bar = full_bar + Cfg::STAGES;
  uint64_t* tfull_bar = empty_bar + Cfg::STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // per-column vectors: staged in smem once per (persistent) CTA instead of a just-in-time __ldg per chunk, which
  // ncu showed as the epilogue's dominant stall (long_scoreboard)
  float* sbias = reinterpret_cast<float*>(smem + Cfg::OFF_VEC);
  float* sgamma = sbias + g.N;
  if (EPI == ACX_EPI_BIAS_GELU_FOLD) {
    // interleaved {b[2q], b[2q+1], s[2q], s[2q+1]}: one 16-byte load per column pair in the folded epilogue
    for (int i = threadIdx.x; i < g.N; i += blockDim.x) {
      sbias[4 * (i >> 1) + (i & 1)] = g.bias[i];
      sbias[4 * (i >> 1) + 2 + (i & 1)] = g.ln_s[i];
    }
  } else {
    for (int i = threadIdx.x; i < g.N; i += blockDim.x) {
      sbias[i] = g.bias[i];
      if (EPI == ACX_EPI_BIAS_SCALE_RESID) sgamma[i] = g.gamma[i];
    }
  }

  if (warp == 0 && ptx::elect_one()) {
    ptx::prefetch_tensormap(&tmA);
    ptx::prefetch_tensormap(&tmB);
    ptx::prefetch_tensormap(&tmOut);
  }
  if (warp == 1 && ptx::elect_one()) {
    for (int s = 0; s < Cfg::STAGES; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tfull_bar[a], 1);
      ptx::mbar_init(&tempty_bar[a], NEPI * CG);   // the leader's copy collects the epilogue warps of both CTAs
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    if (CG == 2) {
      ptx::tmem_alloc_cg2(tmem_slot, Cfg::TMEM_COLS);
      ptx::tmem_relinquish_cg2();
    } else {
      ptx::tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (CG == 2) ptx::cluster_sync_all();            // peer barriers are initialised before any remote arrive / TMA
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_trigger();       // TMEM is ours: the next kernel's CTAs may start their prologue on SMs that free up
  pdl_wait();          // everything above touched only weights; A, the residual and the output belong to earlier kernels

  const int num_m_tiles = (g.M + Cfg::BM * CG - 1) / (Cfg::BM * CG);   // tiles of 128 (CG=1) or 256 (CG=2) rows
  const int num_n_tiles = g.N / BN;
  const int num_tiles = num_m_tiles * num_n_tiles;
  const int num_kb = (g.K + Cfg::BK - 1) / Cfg::BK;

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = unit; tile < num_tiles; tile += num_units) {
        const int tt = g.reverse ? num_tiles - 1 - tile : tile;      // see GemmArgs::reverse
        const int m0 = (tt / num_n_tiles) * Cfg::BM * CG + cta_rank * Cfg::BM;
        const int n0 = (tt % num_n_tiles) * BN + cta_rank * (BN / CG);
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
          uint8_t* sb = sa + Cfg::A_BYTES;
          if (CG == 2) {
            // both CTAs' bytes complete on the LEADER's full barrier; only the leader arms it
            if (cta_rank == 0) ptx::mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
            if (g.a_gp) ptx::tma_load_3d_cg2(sa, &tmA, &full_bar[stage], 0, m0 >> 5, kb * (Cfg::BK / 8));
            else ptx::tma_load_2d_cg2(sa, &tmA, &full_bar[stage], kb * Cfg::BK, m0);
            ptx::tma_load_2d_cg2(sb, &tmB, &full_bar[stage], kb * Cfg::BK, n0);
          } else {
            ptx::mbar_arrive_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
            if (g.a_gp) ptx::tma_load_3d(sa, &tmA, &full_bar[stage], 0, m0 >> 5, kb * (Cfg::BK / 8));
            else ptx::tma_load_2d(sa, &tmA, &full_bar[stage], kb * Cfg::BK, m0);
            ptx::tma_load_2d(sb, &tmB, &full_bar[stage], kb * Cfg::BK, n0);
          }
          if (++stage == Cfg::STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer (leader CTA only when paired) ==================================
    if (cta_rank == 0 && ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::umma_idesc_bf16(Cfg::BM * CG, BN);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = unit; tile < num_tiles; tile += num_units, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        ptx::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * Cfg::ACC_STRIDE;
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(&full_bar[stage], phase);
          ptx::tc_fence_after();
          const uint32_t sa = ptx::smem_u32(smem + stage * Cfg::STAGE_BYTES);
          // planar A: [8 groups][128 rows][16 B] un-swizzled, a K step = two groups = 4 KB further
          const uint64_t da = g.a_gp ? ptx::umma_desc_nosw_kmajor(sa, Cfg::BM * 16, 128) : ptx::umma_desc_sw128_kmajor(sa);
          const uint32_t ka = g.a_gp ? (2 * Cfg::BM * 16) >> 4 : 2;
          const uint64_t db = ptx::umma_desc_sw128_kmajor(sa + Cfg::A_BYTES);
#pragma unroll
          for (int k = 0; k < Cfg::BK / 16; ++k) {
            if (kb * Cfg::BK + k * 16 < g.K) {
              // advance 16 bf16 = 32 B along K inside the 128B swizzle row: +2 in the (addr >> 4) field
              if (CG == 2) ptx::umma_bf16_cg2(d_tmem, da + ka * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
              else ptx::umma_bf16(d_tmem, da + ka * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            }
          }
          // smem slot reusable (in both CTAs when paired) once these MMAs retire
          if (CG == 2) ptx::umma_commit_cg2(&empty_bar[stage]);
          else ptx::umma_commit(&empty_bar[stage]);
          if (++stage == Cfg::STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (CG == 2) ptx::umma_commit_cg2(&tfull_bar[acc]);  // accumulator complete -> epilogue warps of both CTAs
        else ptx::umma_commit(&tfull_bar[acc]);
      }
    }
  } else if (warp >= 4) {
    // ================================ epilogue =====================================
    // Each warp owns 32 accumulator rows (its TMEM lane quadrant) x a set of 32-column chunks.  Per chunk:
    // tcgen05.ld (issued one chunk ahead) -> bias / GELU / gamma*x + residual -> bf16 -> 64B-swizzled smem tile ->
    // one TMA store (coalesced, asynchronous, clipped at M).  The residual tile is fetched with coalesced 16-byte
    // loads (8 rows x 64 B per instruction) one chunk ahead and transposed through smem.
    const int ew = warp - 4;
    const int quad = warp & 3;            // TMEM lane quadrant this warp may access
    const int group = ew >> 2;            // column group
    const int ch_begin = group == 0 ? 0 : Cfg::CH_G0;
    const int ch_count = group == 0 ? Cfg::CH_G0 : Cfg::NCHUNKS - Cfg::CH_G0;
    uint8_t* stg = smem + Cfg::OFF_STG + ew * Cfg::STG_PER_WARP;
    uint8_t* rbuf = stg + 2 * Cfg::STG_TILE;
    const int sw = (lane >> 1) & 3;       // SWIZZLE_64B: 16-byte chunk j of row r lives at chunk j ^ ((r >> 1) & 3)
    const int ld_piece = lane & 3, ld_row = lane >> 2;   // coalesced residual fetch: 4 pieces x 8 rows per instruction
    int it = 0;
    uint32_t store_parity = 0;            // which staging tile the next chunk uses
    for (int tile = unit; tile < num_tiles; tile += num_units, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int tt = g.reverse ? num_tiles - 1 - tile : tile;
      const int m0 = (tt / num_n_tiles) * Cfg::BM * CG + cta_rank * Cfg::BM;
      const int n0 = (tt % num_n_tiles) * BN;
      const int row0 = m0 + quad * 32;
      uint4 rq[4];
      auto fetch_resid = [&](int ci) {
        if (EPI != ACX_EPI_BIAS_SCALE_RESID) return;
        const int n = n0 + (ch_begin + ci) * Cfg::CHUNK;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int r = row0 + ld_row + 8 * q;
          rq[q] = make_uint4(0u, 0u, 0u, 0u);
          if (r < g.M)
            rq[q] = g.out_gp ? *reinterpret_cast<const uint4*>(g.resid + ((size_t)((n >> 3) + ld_piece) * (((size_t)g.M + 127) / 128 * 128) + r) * 8)
                             : *reinterpret_cast<const uint4*>(g.resid + (size_t)r * g.N + n + ld_piece * 8);
        }
      };
      fetch_resid(0);   // overlaps the wait for the accumulator
      LnFold fold{0ull, 0ull, ptx::smem_u32(sbias), ptx::smem_u32(sbias)};
      if (EPI == ACX_EPI_BIAS_GELU_FOLD) {
        const int r = row0 + lane;
        const float2 stt = r < g.M ? __ldg(g.stats + r) : make_float2(0.f, 0.f);
        fold.rstd2 = f2_pack(stt.x, stt.x);
        fold.nmr2 = f2_pack(stt.y, stt.y);
      }
      ptx::mbar_wait(&tfull_bar[acc], acc_phase);
      ptx::tc_fence_after();
      const uint32_t t_base = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * Cfg::ACC_STRIDE +
                              ch_begin * Cfg::CHUNK;
      uint32_t ra[32], rb[32];
      ptx::tmem_ld_32x32b_x32(t_base, ra);
#pragma unroll
      for (int ci = 0; ci < Cfg::CH_G0; ++ci) {
        if (ci < ch_count) {
          uint32_t(&r)[32] = (ci & 1) ? rb : ra;
          ptx::tmem_ld_wait();
          if (ci + 1 < ch_count) {
            ptx::tmem_ld_32x32b_x32(t_base + (ci + 1) * Cfg::CHUNK, (ci & 1) ? ra : rb);
          } else {
            // last TMEM read of this accumulator has landed: hand it back to the MMA warp
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if (CG == 2) ptx::mbar_arrive_leader(&tempty_bar[acc]);
              else ptx::mbar_arrive(&tempty_bar[acc]);
            }
          }
          const int n = n0 + (ch_begin + ci) * Cfg::CHUNK;
          float v[32];
          if (EPI == ACX_EPI_BIAS_GELU_FOLD) {
            float2 o[16];
            bias_gelu_tile16_sp<false, true>(r, sbias + n, o, fold);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              v[2 * j] = o[j].x;
              v[2 * j + 1] = o[j].y;
            }
          } else if (EPI == ACX_EPI_BIAS_GELU) {
            float2 o[16];
            bias_gelu_tile16_sp<false>(r, sbias + n, o);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              v[2 * j] = o[j].x;
              v[2 * j + 1] = o[j].y;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 b4 = *reinterpret_cast<const float4*>(sbias + n + j);
              v[j + 0] = __uint_as_float(r[j + 0]) + b4.x;
              v[j + 1] = __uint_as_float(r[j + 1]) + b4.y;
              v[j + 2] = __uint_as_float(r[j + 2]) + b4.z;
              v[j + 3] = __uint_as_float(r[j + 3]) + b4.w;
            }
          }
          if (EPI == ACX_EPI_BIAS_SCALE_RESID) {
            // transpose the coalesced residual fetch through smem: lane <- its own row
            __syncwarp();   // previous chunk's reads of rbuf are done
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int rr = ld_row + 8 * q;
              *reinterpret_cast<uint4*>(rbuf + rr * 64 + ((ld_piece ^ ((rr >> 1) & 3)) << 4)) = rq[q];
            }
            __syncwarp();
            if (ci + 1 < ch_count) fetch_resid(ci + 1);
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const uint4 q = *reinterpret_cast<const uint4*>(rbuf + lane * 64 + ((j4 ^ sw) << 4));
              const float4 g0 = *reinterpret_cast<const float4*>(sgamma + n + j4 * 8);
              const float4 g1 = *reinterpret_cast<const float4*>(sgamma + n + j4 * 8 + 4);
              const int j = j4 * 8;
              float2 f;
              f = Pair<bf16>::unpack(q.x); v[j + 0] = fmaf(g0.x, v[j + 0], f.x); v[j + 1] = fmaf(g0.y, v[j + 1], f.y);
              f = Pair<bf16>::unpack(q.y); v[j + 2] = fmaf(g0.z, v[j + 2], f.x); v[j + 3] = fmaf(g0.w, v[j + 3], f.y);
              f = Pair<bf16>::unpack(q.z); v[j + 4] = fmaf(g1.x, v[j + 4], f.x); v[j + 5] = fmaf(g1.y, v[j + 5], f.y);
              f = Pair<bf16>::unpack(q.w); v[j + 6] = fmaf(g1.z, v[j + 6], f.x); v[j + 7] = fmaf(g1.w, v[j + 7], f.y);
            }
          }
          // staging tile free?  (the TMA store issued two chunks ago has finished reading it)
          if (lane == 0) ptx::tma_store_wait_read<1>();
          __syncwarp();
          uint8_t* tile_smem = stg + store_parity * Cfg::STG_TILE;
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const int j = j4 * 8;
            uint4 q;
            q.x = Pair<bf16>::pack(v[j + 0], v[j + 1]);
            q.y = Pair<bf16>::pack(v[j + 2], v[j + 3]);
            q.z = Pair<bf16>::pack(v[j + 4], v[j + 5]);
            q.w = Pair<bf16>::pack(v[j + 6], v[j + 7]);
            // planar output: the staging tile is [4 channel groups][32 rows][16 B] (un-swizzled, one 3-D box)
            *reinterpret_cast<uint4*>(g.out_gp ? tile_smem + j4 * 512 + lane * 16 : tile_smem + lane * 64 + ((j4 ^ sw) << 4)) = q;
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (g.out_gp) ptx::tma_store_3d(&tmOut, tile_smem, 0, row0 >> 5, n >> 3);
            else ptx::tma_store_2d(&tmOut, tile_smem, n, row0);
            ptx::tma_store_commit();
          }
          store_parity ^= 1;
        }
      }
    }
    if (lane == 0) ptx::tma_store_wait_read<0>();   // smem must stay valid until the last store has read it
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (CG == 2) ptx::cluster_sync_all();            // the peer may still multicast into / read from this CTA's smem
  if (warp == 2) {
    ptx::tc_fence_after();
    if (CG == 2) ptx::tmem_dealloc_cg2(tmem_base, Cfg::TMEM_COLS);
    else ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int BN, int EPI, int NEPI, int CG>
static int launch_umma_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmOut, const GemmArgs& g,
                            cudaStream_t st) {
  using Cfg = GemmCfg<BN, NEPI, CG>;
  auto kern = umma_gemm_kernel<BN, EPI, NEPI, CG>;
  ACX_SET_MAX_SMEM(kern, Cfg::SMEM_BYTES);
  ACX_CHECK(g.N * (EPI == ACX_EPI_BIAS_SCALE_RESID || EPI == ACX_EPI_BIAS_GELU_FOLD ? 8 : 4) <= Cfg::VEC_BYTES, ACX_ERR_UNSUPPORTED,
            "gemm_bf16: N=%d exceeds the per-column vectors staged in shared memory", g.N);
  int dev = 0, sms = 0;
  ACX_CUDA(cudaGetDevice(&dev));
  ACX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int tiles = ceil_div(g.M, Cfg::BM * CG) * (g.N / BN);      // work units: CTAs (CG=1) or CTA pairs (CG=2)
  const int units = sms / CG;
  ACX_CUDA(launch_pdl(kern, dim3((tiles < units ? tiles : units) * CG), dim3(Cfg::THREADS), Cfg::SMEM_BYTES, st, CG, PDL_GEMM, tmA, tmB,
                      tmOut, g));
  return ACX_OK;
}

// B operand / output maps and tile-shape dispatch.  A CTA pair (CG = 2) is used when there are enough 256-row tiles to
// fill every SM pair (74 on a B200; taken from the device, not assumed); small problems keep one CTA per 128-row tile.
template <int EPI>
static int dispatch_bn(const CUtensorMap& tmA, const void* W, const GemmArgs& g, cudaStream_t st) {
  int bn = 0;
  for (int cand : {256, 192, 128, 96}) {   // the largest supported BN that divides N (fewer A re-reads, longer MMAs)
    if (g.N % cand == 0) {
      bn = cand;
      break;
    }
  }
  ACX_CHECK(bn != 0, ACX_ERR_UNSUPPORTED, "gemm_bf16: N=%d is not a multiple of 96/128/192/256", g.N);
  const long long pairs = sm_count() / 2;     // 74 on a B200
  // Wave quantisation: a persistent grid of `pairs` CTA pairs runs ceil(tiles / pairs) rounds of BN-wide tiles, so when both
  // 256 and 192 divide N the cheaper of  rounds(BN) * BN  wins (ties keep 256: fewer A re-reads).  Stage 3 at 64 clips:
  // N = 768 is 165 tiles = 3 rounds at BN 256 (2.2 needed) but 220 tiles = 3 rounds at BN 192 -- a quarter less work.
  if (bn == 256 && g.N % 192 == 0) {
    const long long mt = ceil_div(g.M, 256);
    const long long r256 = (mt * (g.N / 256) + pairs - 1) / pairs * 256, r192 = (mt * (g.N / 192) + pairs - 1) / pairs * 192;
    if (mt * (g.N / 192) >= pairs && r192 < r256) bn = 192;
  }
  const bool pair = (bn == 256 || bn == 192) && (long long)ceil_div(g.M, 256) * (g.N / bn) >= pairs;
  CUtensorMap tmB;
  int rc = make_tmap_2d_bf16(&tmB, W, (uint64_t)g.K, (uint64_t)g.N, (uint64_t)g.K * 2, 64,
                             (uint32_t)(pair ? bn / 2 : bn));
  if (rc != ACX_OK) return rc;
  // output: 32-column x 32-row boxes (one per epilogue warp and chunk), 64B swizzle
  CUtensorMap tmOut;
  rc = g.out_gp ? make_tmap_gp_bf16(&tmOut, g.out, (uint64_t)g.M, (uint64_t)g.N / 8, 32, 4)
                : make_tmap_2d_bf16(&tmOut, g.out, (uint64_t)g.N, (uint64_t)g.M, (uint64_t)g.N * 2, 32, 32,
                                    CU_TENSOR_MAP_SWIZZLE_64B);
  if (rc != ACX_OK) return rc;
  if (pair) {
    if (bn == 256) return launch_umma_gemm<256, EPI, 8, 2>(tmA, tmB, tmOut, g, st);
    return launch_umma_gemm<192, EPI, 8, 2>(tmA, tmB, tmOut, g, st);
  }
  switch (bn) {
    case 256: return launch_umma_gemm<256, EPI, 8, 1>(tmA, tmB, tmOut, g, st);
    case 192: return launch_umma_gemm<192, EPI, 8, 1>(tmA, tmB, tmOut, g, st);
    case 128: return launch_umma_gemm<128, EPI, 8, 1>(tmA, tmB, tmOut, g, st);
    default:  return launch_umma_gemm<96, EPI, 8, 1>(tmA, tmB, tmOut, g, st);
  }
}

}  // namespace acx

using namespace acx;

static int gemm_bf16_impl(const void* A, const void* W, void* out, int M, int N, int K, int epilogue, const float* bias,
                          const float* gamma, const void* resid, int out_gp, int a_gp, const float* stats,
                          const float* ln_s, void* stream) {
  ACX_CHECK(A && W && out && bias, ACX_ERR_ARG, "gemm_bf16: null pointer (A, W, out and bias are required)");
  ACX_CHECK(M > 0 && N > 0 && K > 0 && K % 8 == 0, ACX_ERR_ARG, "gemm_bf16: K=%d must be a positive multiple of 8", K);
  ACX_CHECK((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0 &&
                (reinterpret_cast<uintptr_t>(out) & 15) == 0,
            ACX_ERR_ARG, "gemm_bf16: A, W and out must be 16-byte aligned");
  if (epilogue == ACX_EPI_BIAS_SCALE_RESID)
    ACX_CHECK(gamma && resid, ACX_ERR_ARG, "gemm_bf16: scale+residual epilogue needs gamma and resid");
  ACX_CHECK(!out_gp || epilogue != ACX_EPI_BIAS_GELU, ACX_ERR_UNSUPPORTED, "gemm_bf16: the hidden activation stays row-major");
  ACX_CHECK(!a_gp || K % 64 == 0, ACX_ERR_UNSUPPORTED, "gemm_bf16: a planar A operand needs K %% 64 == 0 (got %d)", K);
  ACX_CHECK((stats == nullptr) == (ln_s == nullptr), ACX_ERR_ARG, "gemm_bf16: stats and ln_s go together");
  ACX_CHECK(!stats || epilogue == ACX_EPI_BIAS_GELU, ACX_ERR_UNSUPPORTED, "gemm_bf16: the LayerNorm fold belongs to the GELU epilogue");
  GemmArgs g;
  g.out = reinterpret_cast<bf16*>(out);
  g.bias = bias;
  g.gamma = gamma;
  g.resid = reinterpret_cast<const bf16*>(resid);
  g.M = M;
  g.N = N;
  g.K = K;
  g.out_gp = out_gp;
  g.a_gp = a_gp;
  g.stats = reinterpret_cast<const float2*>(stats);
  g.ln_s = ln_s;
  // the pwconv2 GEMMs (residual epilogue) consume what pwconv1 has just written front to back
  g.reverse = epilogue == ACX_EPI_BIAS_SCALE_RESID && (size_t)M * K * 2 > (size_t)96 << 20;
  CUtensorMap tmA;
  int rc = a_gp ? make_tmap_gp_bf16(&tmA, A, (uint64_t)M, (uint64_t)K / 8, 128, 8)
                : make_tmap_2d_bf16(&tmA, A, (uint64_t)K, (uint64_t)M, (uint64_t)K * 2, 64, 128);
  if (rc != ACX_OK) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  switch (epilogue) {
    case ACX_EPI_BIAS: return dispatch_bn<ACX_EPI_BIAS>(tmA, W, g, st);
    case ACX_EPI_BIAS_GELU:
      return stats ? dispatch_bn<ACX_EPI_BIAS_GELU_FOLD>(tmA, W, g, st) : dispatch_bn<ACX_EPI_BIAS_GELU>(tmA, W, g, st);
    case ACX_EPI_BIAS_SCALE_RESID: return dispatch_bn<ACX_EPI_BIAS_SCALE_RESID>(tmA, W, g, st);
    default:
      set_error("gemm_bf16: unknown epilogue %d", epilogue);
      return ACX_ERR_ARG;
  }
}

extern "C" int acx_gemm_bf16(const void* A, const void* W, void* out, int M, int N, int K, int epilogue,
                             const float* bias, const float* gamma, const void* resid, void* stream) {
  return gemm_bf16_impl(A, W, out, M, N, K, epilogue, bias, gamma, resid, 0, 0, nullptr, nullptr, stream);
}

// out = A . W^T + bias written GROUP-PLANAR, [N/8][Mp][8] (Mp = M rounded up to 128): the downsample GEMM in front of a
// stage whose depthwise conv runs on the tensor cores hands over in that layout instead of a transpose pass.
extern "C" int acx_gemm_bf16_gp_out(const void* A, const void* W, void* out, int M, int N, int K, const float* bias,
                                    void* stream) {
  return gemm_bf16_impl(A, W, out, M, N, K, ACX_EPI_BIAS, bias, nullptr, nullptr, 1, 0, nullptr, nullptr, stream);
}

// The two GEMMs of a Block MLP on group-planar activations (stages whose MLP is not the fused kernel):
//   pwconv1: hid = GELU( LN(v) . W1^T + b1 ) with v planar [C/8][Mp][8], the LayerNorm folded (w1 = bf16(W1 ln_w),
//            b1 = b1 + W1 ln_b, ln_s = row sums of w1, stats = acx_gp_row_stats(v)); hid row-major (M, 4C);
//   pwconv2: x += gamma * (hid . W2^T + b2) with x planar, updated in place.
extern "C" int acx_gemm_bf16_pw1_gp(const void* v_gp, const void* w1f, void* hid, int M, int N, int K, const float* b1f,
                                    const float* stats, const float* ln_s, void* stream) {
  ACX_CHECK(stats && ln_s, ACX_ERR_ARG, "gemm_bf16_pw1_gp: stats and ln_s are required");
  return gemm_bf16_impl(v_gp, w1f, hid, M, N, K, ACX_EPI_BIAS_GELU, b1f, nullptr, nullptr, 0, 1, stats, ln_s, stream);
}
extern "C" int acx_gemm_bf16_pw2_gp(const void* hid, const void* w2, void* x_gp, int M, int N, int K, const float* b2,
                                    const float* gamma, void* stream) {
  return gemm_bf16_impl(hid, w2, x_gp, M, N, K, ACX_EPI_BIAS_SCALE_RESID, b2, gamma, x_gp, 1, 0, nullptr, nullptr, stream);
}
