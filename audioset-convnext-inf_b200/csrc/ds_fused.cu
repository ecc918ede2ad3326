// Downsample layer as ONE implicit-GEMM kernel (reference convnext.py:230-235: LayerNorm(channels_first) -> Conv2d(k2, s2)).
//
//   out[p, n] = bias[n] + sum_{dy, dx, c} W[n, c, dy, dx] * LN(x[b, 2 oy + dy, 2 ox + dx, :])[c]        p = (b, oy, ox)
//
// The patch matrix (M/4 x 4C) that `ln_patchify` used to write to HBM and the GEMM read back never exists: the GEMM's A
// operand is produced in shared memory by gather warps that read the group-planar residual stream [C/8][Mp][8], apply the
// per-pixel LayerNorm in registers and store the K-major 128B-swizzled tile the tensor core reads.
//
//   warp 0        TMA producer of the weight tiles (B operand), STAGES-deep ring shared with the gather warps
//   warp 1        MMA issuer (tcgen05.mma M128 N192 K16, NSUB of them per K step: a tile is 128 x 192 or 128 x 384)
//   warp 2        TMEM allocator
//   warps 4..11   gather: per tile (1) statistics -- thread = (output row, dy): sums over the C channels of its two
//                 adjacent source pixels (one 32-byte run per channel group, planes read coalesced across the warp);
//                 (2) per 64-wide K block: 2 x 32 bytes per thread -> (x - mean) rstd ln_w + ln_b -> bf16 -> swizzled
//                 smem; the second read of x hits L1/L2 (HBM sees x once)
//   warps 12..15  epilogue: tcgen05.ld -> + bias -> bf16 -> staging tile -> TMA store (row-major or group-planar)
//
// K is ordered (dy, channel group, dx, 8 channels) -- the host packs the conv weight the same way (engine.py) -- so that
// the two horizontally adjacent source pixels of a patch are 32 contiguous bytes in global memory AND in the operand row.
#include "common.cuh"
#include "ptx.cuh"
#include "tmap.cuh"

namespace acx {
namespace dsf {

struct DsArgs {
  const uint4* x;        // group-planar input, 16-byte pieces: [C/8][Mp_in]
  const float* ln_w;
  const float* ln_b;
  const float* bias;
  long long Mp_in;       // plane stride in pieces (input pixels rounded up to 128)
  int H, W, Ho, Wo;      // input map / output map
  int Mo;                // output rows = B * Ho * Wo
  int out_gp;            // 1: output group-planar [2C/8][Mp_out][8]; 0: row-major (Mo, 2C)
};

template <int C>
struct DsCfg {
  static constexpr int BM = 128, BK = 64, BN = 192;
  static constexpr int N = 2 * C, K = 4 * C;
  static constexpr int NSUB = C == 96 ? 1 : 2;             // N = 192 MMAs per K step
  static constexpr int TILE_N = NSUB * BN;                 // 192 / 384 / 384
  static constexpr int N_TILES = N / TILE_N;               // 1 / 1 / 2
  static constexpr int NKB = K / BK;                       // 6 / 12 / 24
  static constexpr int KB_PER_DY = C / 32;                 // K blocks per source row of the patch
  static constexpr int G = C / 8;                          // channel groups (planes)
  static constexpr int A_BYTES = BM * BK * 2;              // 16 KB
  static constexpr int B_SUB = BN * BK * 2;                // 24 KB
  static constexpr int B_BYTES = NSUB * B_SUB;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;    // 40 / 64 KB
  static constexpr int STAGES = NSUB == 1 ? 4 : 3;
  static constexpr int NACC = NSUB == 1 ? 2 : 1;           // accumulator buffers in TMEM
  static constexpr int ACC_STRIDE = 256;
  static constexpr int TMEM_COLS = 512;
  static constexpr int NGATHER = 8, NEPI = 4;              // warps
  static constexpr int THREADS = 128 + 32 * (NGATHER + NEPI);
  static constexpr int NCHUNKS = TILE_N / 32;
  static constexpr int STG_TILE = 32 * 32 * 2;             // 32 rows x 32 columns bf16
  static constexpr int OFF_STG = STAGES * STAGE_BYTES;
  static constexpr int OFF_STATS = OFF_STG + NEPI * 2 * STG_TILE;
  static constexpr int OFF_VEC = OFF_STATS + 2 * BM * 4 * 8;           // [2][128 rows][4 source pixels] (mean, rstd)
  static constexpr int OFF_BAR = OFF_VEC + (2 * C + N) * 4;            // ln_w[C], ln_b[C], bias[N]
  static constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024 /*align*/;
  static_assert(N % TILE_N == 0 && K % BK == 0 && C % 32 == 0, "shape");
  static_assert(B_SUB % 1024 == 0 && STAGE_BYTES % 1024 == 0, "swizzle atoms");
  static_assert(NACC * ACC_STRIDE <= TMEM_COLS && TILE_N <= TMEM_COLS, "TMEM");
  static_assert(SMEM_BYTES <= 227 * 1024, "smem budget");
};

// The two horizontally adjacent source pixels of a patch (one channel group) are 32 contiguous, 32-byte aligned bytes: ONE
// 256-bit load (LDG.256, sm_100).  Two 16-byte loads with a 32-byte lane stride made every warp instruction touch 32
// half-used sectors, twice.
__device__ __forceinline__ void ldg256(const uint4* p, uint4& lo, uint4& hi) {
  unsigned long long a, b, c, d;
  asm volatile("ld.global.nc.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
  lo = make_uint4((uint32_t)a, (uint32_t)(a >> 32), (uint32_t)b, (uint32_t)(b >> 32));
  hi = make_uint4((uint32_t)c, (uint32_t)(c >> 32), (uint32_t)d, (uint32_t)(d >> 32));
}

// Explicit shared-space accesses.  Through generic pointers the compiler emitted LD.E / ST.E for the statistics, the LayerNorm
// vectors and the operand stores; a generic load is tracked by the same long scoreboard as the global loads in flight, so the
// first one of a K block waited for the loads issued a moment earlier for the NEXT block (ncu: the kernel's top stall).
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float2 lds64(uint32_t addr) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts64(uint32_t addr, const float2& v) {
  asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(v.x), "f"(v.y) : "memory");
}

__device__ __forceinline__ void unpack8(const uint4 v, float (&f)[8]) {
  float2 t;
  t = Pair<bf16>::unpack(v.x); f[0] = t.x; f[1] = t.y;
  t = Pair<bf16>::unpack(v.y); f[2] = t.x; f[3] = t.y;
  t = Pair<bf16>::unpack(v.z); f[4] = t.x; f[5] = t.y;
  t = Pair<bf16>::unpack(v.w); f[6] = t.x; f[7] = t.y;
}

template <int C>
__global__ void __launch_bounds__(DsCfg<C>::THREADS, 1)
    ds_fused_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmOut, DsArgs a) {
  using Cfg = DsCfg<C>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* empty_bar = full_bar + Cfg::STAGES;
  uint64_t* tfull_bar = empty_bar + Cfg::STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  float* slnw = reinterpret_cast<float*>(smem + Cfg::OFF_VEC);
  float* slnb = slnw + C;
  float* sbias = slnb + C;
  float2* sstat = reinterpret_cast<float2*>(smem + Cfg::OFF_STATS);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    slnw[i] = a.ln_w[i];
    slnb[i] = a.ln_b[i];
  }
  for (int i = threadIdx.x; i < Cfg::N; i += blockDim.x) sbias[i] = a.bias[i];
  if (warp == 0 && ptx::elect_one()) {
    ptx::prefetch_tensormap(&tmW);
    ptx::prefetch_tensormap(&tmOut);
  }
  if (warp == 1 && ptx::elect_one()) {
    for (int s = 0; s < Cfg::STAGES; ++s) {
      ptx::mbar_init(&full_bar[s], 1 + Cfg::NGATHER);     // weight producer (with the TMA bytes) + one arrive per gather warp
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&tfull_bar[i], 1);
      ptx::mbar_init(&tempty_bar[i], Cfg::NEPI);
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
  pdl_trigger();                  // programmatic dependent launch (common.cuh): TMEM is allocated
  if (warp != 0) pdl_wait();      // the weight producer touches only weights and may run ahead of the previous kernel

  const int num_m_tiles = (a.Mo + Cfg::BM - 1) / Cfg::BM;
  const int num_tiles = num_m_tiles * Cfg::N_TILES;

  if (warp == 0) {
    // ================================ weight (B operand) producer ================================
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int n0 = (tile % Cfg::N_TILES) * Cfg::TILE_N;
        for (int kb = 0; kb < Cfg::NKB; ++kb) {
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sb = smem + stage * Cfg::STAGE_BYTES + Cfg::A_BYTES;
          ptx::mbar_arrive_expect_tx(&full_bar[stage], Cfg::B_BYTES);
#pragma unroll
          for (int s = 0; s < Cfg::NSUB; ++s)
            ptx::tma_load_2d(sb + s * Cfg::B_SUB, &tmW, &full_bar[stage], kb * Cfg::BK, n0 + s * Cfg::BN);
          if (++stage == Cfg::STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    if (ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::umma_idesc_bf16(Cfg::BM, Cfg::BN);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
        const int acc = Cfg::NACC == 2 ? (it & 1) : 0;
        const uint32_t acc_phase = Cfg::NACC == 2 ? ((it >> 1) & 1) : (it & 1);
        ptx::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * Cfg::ACC_STRIDE;
        for (int kb = 0; kb < Cfg::NKB; ++kb) {
          ptx::mbar_wait(&full_bar[stage], phase);
          ptx::tc_fence_after();
          const uint32_t sa = ptx::smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint64_t da = ptx::umma_desc_sw128_kmajor(sa);
#pragma unroll
          for (int k = 0; k < Cfg::BK / 16; ++k) {
#pragma unroll
            for (int s = 0; s < Cfg::NSUB; ++s) {
              const uint64_t db = ptx::umma_desc_sw128_kmajor(sa + Cfg::A_BYTES + s * Cfg::B_SUB);
              ptx::umma_bf16(d_tmem + s * Cfg::BN, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            }
          }
          ptx::umma_commit(&empty_bar[stage]);
          if (++stage == Cfg::STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        ptx::umma_commit(&tfull_bar[acc]);
      }
    }
  } else if (warp >= 4 && warp < 4 + Cfg::NGATHER) {
    // ================================ gather + LayerNorm: the A operand ================================
    const int t = threadIdx.x - 128;          // 0..255
    const int r = t & 127;                    // output row of the tile
    const int hs = t >> 7;                    // statistics: dy; operand: which half of the K block's four channel groups
    const uint32_t sw = static_cast<uint32_t>(r & 7);
    const uint32_t smem_a = ptx::smem_u32(smem), sstat_a = ptx::smem_u32(sstat), slnw_a = ptx::smem_u32(slnw), slnb_a = ptx::smem_u32(slnb);
    // source pixel (dy = 0, dx = 0) of output row r of a tile, as a piece index into plane 0
    auto tile_src = [&](int tile, bool& valid) -> const uint4* {
      const int p = (tile / Cfg::N_TILES) * Cfg::BM + r;
      valid = tile < num_tiles && p < a.Mo;
      const int pp = valid ? p : 0;
      const int ox = pp % a.Wo;
      const int oy = (pp / a.Wo) % a.Ho;
      const int b = pp / (a.Wo * a.Ho);
      return a.x + ((long long)b * a.H + 2 * oy) * a.W + 2 * ox;
    };
    // ---- statistics of this thread's two source pixels (row 2 oy + hs, columns 2 ox and 2 ox + 1): shifted single-pass sums
    float2 s0, q0, s1, q1, n0, n1;
    float sh0 = 0.f, sh1 = 0.f;
    auto stats_reset = [&](const uint4& f0, const uint4& f1, bool valid) {
      s0 = q0 = s1 = q1 = make_float2(0.f, 0.f);
      sh0 = valid ? __uint_as_float(f0.x << 16) : 0.f;      // shift = the pixel's first channel
      sh1 = valid ? __uint_as_float(f1.x << 16) : 0.f;
      n0 = make_float2(-sh0, -sh0);
      n1 = make_float2(-sh1, -sh1);
    };
    auto stats_add = [&](const uint4& u0, const uint4& u1) {
      const uint32_t w0[4] = {u0.x, u0.y, u0.z, u0.w};
      const uint32_t w1[4] = {u1.x, u1.y, u1.z, u1.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 d0 = __fadd2_rn(Pair<bf16>::unpack(w0[k]), n0);
        const float2 d1 = __fadd2_rn(Pair<bf16>::unpack(w1[k]), n1);
        s0 = __fadd2_rn(s0, d0);
        q0 = __ffma2_rn(d0, d0, q0);
        s1 = __fadd2_rn(s1, d1);
        q1 = __ffma2_rn(d1, d1, q1);
      }
    };
    auto stats_store = [&](uint32_t st) {
      const float inv_c = 1.0f / C;
      const float md0 = (s0.x + s0.y) * inv_c, md1 = (s1.x + s1.y) * inv_c;
      const float v0 = fmaxf((q0.x + q0.y) * inv_c - md0 * md0, 0.f), v1 = fmaxf((q1.x + q1.y) * inv_c - md1 * md1, 0.f);
      sts64(st + (r * 4 + hs * 2 + 0) * 8, make_float2(md0 + sh0, rsqrtf(v0 + 1e-6f)));     // channels_first LayerNorm, eps 1e-6 (CX:231)
      sts64(st + (r * 4 + hs * 2 + 1) * 8, make_float2(md1 + sh1, rsqrtf(v1 + 1e-6f)));
    };
    // L2 prefetch of this thread's share (row r, source row hs, channel groups 2 j and 2 j + 1: two 32-byte sectors) of a
    // tile.  The register-held loads below keep only ~32 KB per SM in flight, a third of what the HBM latency needs; the
    // prefetches cost no registers and run a whole tile (two at start-up) ahead of the loads, which then hit L2.
    auto prefetch_part = [&](const uint4* tsrc0, bool v, int j) {
      if (v) {
        const uint4* q = tsrc0 + hs * a.W + (long long)(2 * j) * a.Mp_in;
        ptx::prefetch_l2(q);
        ptx::prefetch_l2(q + a.Mp_in);
      }
    };
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    bool valid;
    const uint4* src0 = tile_src(blockIdx.x, valid);
    {
      bool v1;
      const uint4* t1 = tile_src(blockIdx.x + gridDim.x, v1);
      for (int j = 0; j < Cfg::NKB; ++j) prefetch_part(src0, valid, j);
      for (int j = 0; j < Cfg::NKB; ++j) prefetch_part(t1, v1, j);
    }
    {
      // first tile of this CTA: all channel groups at once, 12 independent 16-byte loads in flight per thread
      const uint4* px = src0 + hs * a.W;
      const uint4 z = make_uint4(0u, 0u, 0u, 0u);
      uint4 f0 = z, f1 = z;
      if (valid) ldg256(px, f0, f1);
      stats_reset(f0, f1, valid);
      if (valid) {
        constexpr int U = 6;
#pragma unroll 1
        for (int g0 = 0; g0 < Cfg::G; g0 += U) {
          uint4 u0[U], u1[U];
#pragma unroll
          for (int j = 0; j < U; ++j) ldg256(px + (long long)(g0 + j) * a.Mp_in, u0[j], u1[j]);
#pragma unroll
          for (int j = 0; j < U; ++j) stats_add(u0[j], u1[j]);
        }
      }
      stats_store(sstat_a);
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");          // the gather warps only: statistics of the tile are complete
    // operand loads of one K block: (dy, four channel groups); this thread: row r, groups 2 hs and 2 hs + 1, both dx
    auto load_kb = [&](const uint4* tsrc0, bool v, int kb, uint4 (&d)[4]) {
      const int dy = kb / Cfg::KB_PER_DY;
      const int g = (kb - dy * Cfg::KB_PER_DY) * 4 + 2 * hs;
      const uint4* px = tsrc0 + dy * a.W + (long long)g * a.Mp_in;
      if (v) {
        ldg256(px, d[0], d[1]);
        ldg256(px + a.Mp_in, d[2], d[3]);
      } else {
        d[0] = d[1] = d[2] = d[3] = make_uint4(0u, 0u, 0u, 0u);
      }
    };
    uint4 buf_a[4], buf_b[4];
    load_kb(src0, valid, 0, buf_a);
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const uint32_t st = sstat_a + (it & 1) * (Cfg::BM * 4 * 8);
      // The NEXT tile's statistics ride along with this tile's K blocks: two channel groups per block (G / NKB = 2), the
      // loads issued one block ahead of their use.  They are what pulls x from HBM (into L2 for the operand pass of the next
      // tile) while this tile is being normalised -- a stand-alone statistics phase per tile left the tensor core and HBM
      // idle for a DRAM round trip per six groups.
      bool nvalid;
      const uint4* nsrc0 = tile_src(tile + gridDim.x, nvalid);
      const bool has_next = tile + (int)gridDim.x < num_tiles;
      bool v2;
      const uint4* t2 = tile_src(tile + 2 * gridDim.x, v2);
      const uint4* npx = nsrc0 + hs * a.W;
      uint4 sp[4];
      auto stats_issue = [&](int j) {
        const uint4* q = npx + (long long)(2 * j) * a.Mp_in;
        if (nvalid) {
          ldg256(q, sp[0], sp[1]);
          ldg256(q + a.Mp_in, sp[2], sp[3]);
        } else {
          sp[0] = sp[1] = sp[2] = sp[3] = make_uint4(0u, 0u, 0u, 0u);
        }
      };
      // The operand loads run one K block ahead -- across the tile boundary too -- in two register buffers that trade roles
      // (the loop is unrolled by two; copying `nxt` into `cur` at the end of an iteration made every block wait for the
      // loads it had just issued: ncu source view, the MOV after the stores was the kernel's top stall).
      auto step = [&](const int kb, uint4 (&cur)[4], uint4 (&nxt)[4]) {
        prefetch_part(t2, v2, kb);
        if (has_next) {
          if (kb == 1) stats_reset(sp[0], sp[1], nvalid);
          if (kb > 0) {
            stats_add(sp[0], sp[1]);
            stats_add(sp[2], sp[3]);
          }
          stats_issue(kb);
        }
        if (kb + 1 < Cfg::NKB) load_kb(src0, valid, kb + 1, nxt);
        else if (has_next) load_kb(nsrc0, nvalid, 0, nxt);
        const int dy = kb / Cfg::KB_PER_DY;
        const int g = (kb - dy * Cfg::KB_PER_DY) * 4 + 2 * hs;
        // packed fp32x2 arithmetic (FADD2 / FMUL2 / FFMA2): ((x - mean) rstd) ln_w + ln_b, two channels per instruction.  Rows past
        // the last output pixel carry zeros and finite statistics: their (finite) results are clipped by the store.
        float2 nm[2], rs[2];
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
          const float2 sx = lds64(st + (r * 4 + dy * 2 + dx) * 8);
          nm[dx] = make_float2(-sx.x, -sx.x);
          rs[dx] = make_float2(sx.y, sx.y);
        }
        uint4 o[4];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const float4 w0 = lds128(slnw_a + (g + u) * 32), w1 = lds128(slnw_a + (g + u) * 32 + 16);
          const float4 b0 = lds128(slnb_a + (g + u) * 32), b1 = lds128(slnb_a + (g + u) * 32 + 16);
          const float2 gw[4] = {make_float2(w0.x, w0.y), make_float2(w0.z, w0.w), make_float2(w1.x, w1.y), make_float2(w1.z, w1.w)};
          const float2 gb[4] = {make_float2(b0.x, b0.y), make_float2(b0.z, b0.w), make_float2(b1.x, b1.y), make_float2(b1.z, b1.w)};
#pragma unroll
          for (int dx = 0; dx < 2; ++dx) {
            const uint4 c4 = cur[u * 2 + dx];
            const uint32_t wv[4] = {c4.x, c4.y, c4.z, c4.w};
            uint32_t ov[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              float2 f = __fmul2_rn(__fadd2_rn(Pair<bf16>::unpack(wv[j]), nm[dx]), rs[dx]);
              f = __ffma2_rn(f, gw[j], gb[j]);
              ov[j] = Pair<bf16>::pack(f.x, f.y);
            }
            o[u * 2 + dx] = make_uint4(ov[0], ov[1], ov[2], ov[3]);
          }
        }
        ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
        const uint32_t row = smem_a + stage * Cfg::STAGE_BYTES + r * 128;
#pragma unroll
        for (int i = 0; i < 4; ++i)      // 16-byte slot (2 hs + u) * 2 + dx of the 128-byte row, SWIZZLE_128B: slot ^ (row & 7)
          sts128(row + (((uint32_t)(hs * 4 + i) ^ sw) << 4), o[i]);
        ptx::fence_proxy_async_smem();   // generic-proxy stores -> visible to the tensor core's async-proxy reads
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&full_bar[stage]);
        if (++stage == Cfg::STAGES) {
          stage = 0;
          phase ^= 1;
        }
      };
      static_assert(Cfg::NKB % 2 == 0, "the K loop is unrolled by two");
#pragma unroll 1
      for (int kb = 0; kb < Cfg::NKB; kb += 2) {
        step(kb, buf_a, buf_b);
        step(kb + 1, buf_b, buf_a);
      }
      if (has_next) {
        stats_add(sp[0], sp[1]);
        stats_add(sp[2], sp[3]);
        stats_store(sstat_a + ((it + 1) & 1) * (Cfg::BM * 4 * 8));
        asm volatile("bar.sync 1, 256;" ::: "memory");      // next tile's statistics complete; this tile's no longer read
      }
      src0 = nsrc0;
      valid = nvalid;
    }
  } else if (warp >= 4 + Cfg::NGATHER) {
    // ================================ epilogue ================================
    const int ew = warp - 4 - Cfg::NGATHER;
    const int quad = warp & 3;                 // TMEM lane quadrant this warp may access (warps 12..15 -> 0..3)
    uint8_t* stg = smem + Cfg::OFF_STG + ew * 2 * Cfg::STG_TILE;
    const int swz = (lane >> 1) & 3;           // SWIZZLE_64B of the row-major staging tile
    const uint32_t sbias_a = ptx::smem_u32(sbias);
    int it = 0;
    uint32_t store_parity = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int acc = Cfg::NACC == 2 ? (it & 1) : 0;
      const uint32_t acc_phase = Cfg::NACC == 2 ? ((it >> 1) & 1) : (it & 1);
      const int m0 = (tile / Cfg::N_TILES) * Cfg::BM;
      const int n0 = (tile % Cfg::N_TILES) * Cfg::TILE_N;
      const int row0 = m0 + quad * 32;
      ptx::mbar_wait(&tfull_bar[acc], acc_phase);
      ptx::tc_fence_after();
      const uint32_t t_base = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * Cfg::ACC_STRIDE;
      uint32_t ra[32], rb[32];
      ptx::tmem_ld_32x32b_x32(t_base, ra);
#pragma unroll
      for (int ci = 0; ci < Cfg::NCHUNKS; ++ci) {
        uint32_t(&rr)[32] = (ci & 1) ? rb : ra;
        ptx::tmem_ld_wait();
        if (ci + 1 < Cfg::NCHUNKS) {
          ptx::tmem_ld_32x32b_x32(t_base + (ci + 1) * 32, (ci & 1) ? ra : rb);
        } else {
          ptx::tc_fence_before();            // last TMEM read of this accumulator has landed: hand it back to the MMA warp
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&tempty_bar[acc]);
        }
        const int n = n0 + ci * 32;
        if (lane == 0) ptx::tma_store_wait_read<1>();     // the store issued two chunks ago has finished reading its tile
        __syncwarp();
        uint8_t* tile_smem = stg + store_parity * Cfg::STG_TILE;
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const int j = j4 * 8;
          const float4 b0 = lds128(sbias_a + (n + j) * 4), b1 = lds128(sbias_a + (n + j) * 4 + 16);
          uint4 q;
          q.x = Pair<bf16>::pack(__uint_as_float(rr[j + 0]) + b0.x, __uint_as_float(rr[j + 1]) + b0.y);
          q.y = Pair<bf16>::pack(__uint_as_float(rr[j + 2]) + b0.z, __uint_as_float(rr[j + 3]) + b0.w);
          q.z = Pair<bf16>::pack(__uint_as_float(rr[j + 4]) + b1.x, __uint_as_float(rr[j + 5]) + b1.y);
          q.w = Pair<bf16>::pack(__uint_as_float(rr[j + 6]) + b1.z, __uint_as_float(rr[j + 7]) + b1.w);
          // planar output: [4 channel groups][32 rows][16 B] (one 3-D box); row-major: 32 rows x 64 B, 64B-swizzled
          sts128(ptx::smem_u32(tile_smem) + (a.out_gp ? j4 * 512 + lane * 16 : lane * 64 + ((j4 ^ swz) << 4)), q);
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          if (a.out_gp) ptx::tma_store_3d(&tmOut, tile_smem, 0, row0 >> 5, n >> 3);
          else ptx::tma_store_2d(&tmOut, tile_smem, n, row0);
          ptx::tma_store_commit();
        }
        store_parity ^= 1;
      }
    }
    if (lane == 0) ptx::tma_store_wait_read<0>();   // smem must stay valid until the last store has read it
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int C>
static int launch(const void* x, const float* ln_w, const float* ln_b, const void* w, const float* bias, void* out, int B,
                  int H, int W, int out_gp, cudaStream_t st) {
  using Cfg = DsCfg<C>;
  DsArgs a;
  a.x = reinterpret_cast<const uint4*>(x);
  a.ln_w = ln_w;
  a.ln_b = ln_b;
  a.bias = bias;
  a.Mp_in = (long long)gp_rows_pad((uint64_t)B * H * W);
  a.H = H;
  a.W = W;
  a.Ho = H / 2;
  a.Wo = W / 2;
  a.Mo = B * a.Ho * a.Wo;
  a.out_gp = out_gp;
  CUtensorMap tmW, tmOut;
  int rc = make_tmap_2d_bf16(&tmW, w, (uint64_t)Cfg::K, (uint64_t)Cfg::N, (uint64_t)Cfg::K * 2, 64, Cfg::BN);
  if (rc != ACX_OK) return rc;
  rc = out_gp ? make_tmap_gp_bf16(&tmOut, out, (uint64_t)a.Mo, (uint64_t)Cfg::N / 8, 32, 4)
              : make_tmap_2d_bf16(&tmOut, out, (uint64_t)Cfg::N, (uint64_t)a.Mo, (uint64_t)Cfg::N * 2, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B);
  if (rc != ACX_OK) return rc;
  auto kern = ds_fused_kernel<C>;
  ACX_SET_MAX_SMEM(kern, Cfg::SMEM_BYTES);
  const int tiles = ceil_div(a.Mo, Cfg::BM) * Cfg::N_TILES;
  const int sms = sm_count();
  ACX_CUDA(launch_pdl(kern, dim3(tiles < sms ? tiles : sms), dim3(Cfg::THREADS), Cfg::SMEM_BYTES, st, 1, PDL_GEMM, tmW, tmOut, a));
  return ACX_OK;
}

}  // namespace dsf
}  // namespace acx

using namespace acx;

// x: group-planar bf16 [C/8][Mp][8] (Mp = B*H*W rounded up to 128); w: (2C, 4C) bf16 with k = ((dy * C/8 + g) * 2 + dx) * 8 + c8
// (engine.pack_downsample_weight); out: (B*(H/2)*(W/2), 2C) bf16 row-major, or group-planar when out_gp.
extern "C" int acx_downsample_fused_gp(const void* x, const float* ln_w, const float* ln_b, const void* w, const float* bias,
                                       void* out, int B, int H, int W, int C, int out_gp, void* stream) {
  ACX_CHECK(x && ln_w && ln_b && w && bias && out, ACX_ERR_ARG, "downsample_fused_gp: null pointer");
  ACX_CHECK(B > 0 && H >= 2 && W >= 2 && W % 2 == 0, ACX_ERR_ARG, "downsample_fused_gp: bad shape B=%d H=%d W=%d (W must be even)", B, H, W);
  ACX_CHECK(((reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(out)) & 15) == 0 && (reinterpret_cast<uintptr_t>(x) & 31) == 0,
            ACX_ERR_ARG, "downsample_fused_gp: w and out must be 16-byte aligned, x 32-byte aligned (256-bit loads)");
  ACX_CHECK((long long)B * H * W < (1ll << 31), ACX_ERR_ARG, "downsample_fused_gp: too many pixels");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  switch (C) {
    case 96: return dsf::launch<96>(x, ln_w, ln_b, w, bias, out, B, H, W, out_gp, st);
    case 192: return dsf::launch<192>(x, ln_w, ln_b, w, bias, out, B, H, W, out_gp, st);
    case 384: return dsf::launch<384>(x, ln_w, ln_b, w, bias, out, B, H, W, out_gp, st);
    default:
      set_error("downsample_fused_gp: C=%d not supported (96 / 192 / 384)", C);
      return ACX_ERR_UNSUPPORTED;
  }
}
