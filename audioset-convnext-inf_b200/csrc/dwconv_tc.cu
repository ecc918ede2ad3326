// Depthwise 7x7 convolution on the tcgen05 tensor cores (reference convnext.py:76, the `dwconv` of every Block), bf16 mode.
//
// Why: the CUDA-core kernel (kernels_bw.cu, dwconv_ln) does 49 FMA per element and sits on the FMA pipe: ~123 FMA / clk /
// SM whatever the operand format (tools/ubench/pipes_half.cu: HFMA2 = 63 instr-lanes = the same 126 FMA / clk / SM as
// FFMA, so packed half precision buys nothing on sm_100), i.e. >= 0.118 ms for a stage-0 layer of 64 clips at 100 % pipe
// utilisation.  The tensor pipe does the same layer in ~0.05 ms of MMA time as a banded-Toeplitz GEMM.
//
// Formulation, per channel c and kernel row dy:   D_c[h, w] += sum_k A_c[h + dy, k] * T_{c,dy}[w, k]
//   A_c  = the channel's image rows as a K-major 128B-swizzled smem tile (row = image row, k = image column).  The SAME
//          tile is read at the 7 row offsets dy by advancing the descriptor start address by dy * 128 B (the swizzle is a
//          function of the absolute smem address: tools/ubench/umma_rowshift.cu, dwtc_probe.cu), so it is staged once;
//   T    = 32 x 32 band matrix, T[n, k] = tap[dy][k - n + 3] (7 diagonals), 64B-swizzled.  A 56-wide row is covered by two
//          32-column K windows: the left half (output columns 0..27) reads image columns [0, 32), the right half reads
//          [24, 56) (descriptor start + 48 B) and produces output column 24 + n in accumulator column n (n = 4..31), which
//          makes ONE band matrix serve both halves.  N = 32 instead of 64 keeps K at 32: 2 x 14 MMAs of M64 N32 K16
//          (24.5 clk each, measured: the MMA streams its operands out of smem at 128 B / clk) instead of 28 of N64.
//   D_c  = 64 rows (TMEM lanes) x 32 columns fp32; 8 channels = 256 TMEM columns.
// Unit of work = (clip, 63-row tile, 8-channel group, half): 8 channels because 8 bf16 = 16 B is the smallest piece of an
// NHWC pixel that loads / stores efficiently.  NHWC -> channel-planar happens on the way into smem: each lane loads the
// (pixel, channel-pair) word of an 8 x 8 fragment and stmatrix.trans writes 8 pixels of one channel as one 16-byte row
// (the per-channel tile stride is 73 rows, == 1 mod 8, so the 8 rows of a matrix land in 8 different swizzle positions:
// conflict-free).  The accumulators come back through tcgen05.ld with thread = image row, 8 channels x 8 pixels at a
// time, get the conv bias, and leave as 16-byte NHWC stores.
// Two CTAs per SM (105 KB smem, 256 TMEM columns, <= 128 registers each): the phases of a CTA run one after the other
// (stage, band build / MMA ring, write-out) and the co-resident CTA fills the pipes meanwhile.
//
// LayerNorm is NOT done here: a CTA only ever sees 8 of the C channels of a pixel.  It is applied by
// acx_layernorm_rows (below, one HBM-bound pass, in place) -- or folded into the consumer GEMM's epilogue.
#include <stdlib.h>

#include "common.cuh"
#include "ptx.cuh"

namespace acx {
namespace dwtc {

constexpr int TR = 63;                    // output rows per tile (M = 64; lane 63 is never valid)
constexpr int AR = TR + 6;                // image rows staged per tile
constexpr int A_STRIDE = 73 * 128;        // bytes between the channels' tiles: 73 rows (== 1 mod 8), 9344 B
constexpr int CG = 8;                     // channels per unit
constexpr int BAND_TILE = 32 * 64;        // one dy: 32 rows x 32 k, SWIZZLE_64B
constexpr int BAND = 7 * BAND_TILE;       // one channel
constexpr int NSLOT = 2;
constexpr int THREADS = 256;
constexpr int OFF_A = 0;
constexpr int OFF_BAND = CG * A_STRIDE;                 // 74752 = 73 * 1024
constexpr int OFF_TAPS = OFF_BAND + NSLOT * BAND;       // 8 x 49 bf16 (+ pad)
constexpr int OFF_DUMMY = OFF_TAPS + 1024;              // 32 x 16 B sink for the unused rows of the last stmatrix
constexpr int OFF_BAR = OFF_DUMMY + 512;
constexpr int SMEM_BYTES = OFF_BAR + 128 + 1024;        // + alignment slack
static_assert(OFF_BAND % 1024 == 0 && BAND % 1024 == 0, "swizzle atoms");
static_assert(2 * (SMEM_BYTES + 1024) <= 227 * 1024, "two CTAs per SM");
static_assert(TR * 28 * 16 <= NSLOT * BAND, "the write-out staging of the planar layout lives in the band slots");

__device__ __forceinline__ void stmatrix_x4_trans(uint32_t addr, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
  asm volatile("stmatrix.sync.aligned.m8n8.x4.trans.shared.b16 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(r0), "r"(r1),
               "r"(r2), "r"(r3)
               : "memory");
}
__device__ __forceinline__ uint32_t ldg_nc_u32(const void* p) {
  uint32_t v;
  asm volatile("ld.global.nc.b32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}

// W = image width of the stage (56 / 28 / 14 / 7; <= 32 uses one K window).  x and v are NHWC.
// RAG = ragged batch: clip n has valid[n] rows (clamped to [0, H]); the rows past it are staged as the conv's zero padding,
// so its first valid[n] output rows equal a run at that height (the rows past it are computed but carry no meaning).
template <int W, bool RAG = false>
__global__ void __launch_bounds__(THREADS, 2)
    dwconv_tc_kernel(const bf16* __restrict__ x, const bf16* __restrict__ taps /*[49][C]*/,
                     const float* __restrict__ bias, bf16* __restrict__ v, int n_clips, int H, int C,
                     const int32_t* __restrict__ valid) {
  constexpr int NHALF = W > 32 ? 2 : 1;
  constexpr int WB = (W + 7) / 8;               // 8-pixel blocks per image row
  constexpr int NM = AR * WB;                   // 8 x 8 fragments per unit
  constexpr int NG = (NM + 3) / 4;              // stmatrix.x4 groups
  constexpr int ROUNDS = (NG + 8 * 4 - 1) / (8 * 4);   // per warp: rounds of 4 groups (16 loads in flight per lane)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t s_base = ptx::smem_u32(smem);
  uint16_t* taps_s = reinterpret_cast<uint16_t*>(smem + OFF_TAPS);     // [8][49]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* band_full = bars;           // [NSLOT]  builders -> MMA
  uint64_t* band_empty = bars + 2;      // [NSLOT]  MMA (tcgen05.commit) -> builders
  uint64_t* d_full = bars + 4;          // all MMAs of a half have completed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  // zero once: K padding of the A tiles (columns >= W, rows 69..72) and everything off the band diagonals never change
  for (int i = tid; i < OFF_TAPS / 16; i += THREADS) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  if (tid == 0) {
    for (int s = 0; s < NSLOT; ++s) {
      ptx::mbar_init(&band_full[s], 7);
      ptx::mbar_init(&band_empty[s], 1);
    }
    ptx::mbar_init(d_full, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 0) {
    ptx::tmem_alloc(tmem_slot, 256);
    ptx::tmem_relinquish();
  }
  ptx::fence_proxy_async_smem();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  // band builders (warps 1..7 = 224 threads): thread = (n, dx), writes tap[dy][dx] of the current channel at [n][k = n + dx - 3]
  const int bj = tid - 32;
  const int bn = bj / 7, bdx = bj - bn * 7, bk = bn + bdx - 3;
  const bool b_ok = warp >= 1 && bk >= 0 && bk < 32;
  const uint32_t b_off = bn * 64 + ((((bk >> 3) ^ ((bn >> 1) & 3)) << 4) + ((bk & 7) << 1));

  const int tiles = (H + TR - 1) / TR, groups = C / CG;
  const int units = n_clips * tiles * groups;
  uint32_t bc = 0;          // band-slot uses so far (the MMA thread and the builders count the same sequence)
  uint32_t dphase = 0;
  for (int unit = blockIdx.x; unit < units; unit += gridDim.x) {
    const int g = unit % groups, t = (unit / groups) % tiles, n = unit / (groups * tiles);
    const int h0 = t * TR, c0 = g * CG;
    // ---- taps of the 8 channels -> smem [c][49] -------------------------------------------------------------------
    for (int i = tid; i < 49 * CG; i += THREADS) {
      const int tap = i >> 3, c = i & 7;
      taps_s[c * 49 + tap] = reinterpret_cast<const uint16_t*>(taps)[tap * C + c0 + c];
    }
    // ---- stage: NHWC -> channel-planar A tiles ------------------------------------------------------------------------
    {
      const bf16* xin = x + (size_t)n * H * W * C + c0 + 2 * (lane & 3);
      const int px = lane >> 2;                           // pixel of the fragment this lane loads
      const int sj = lane & 7, smi = lane >> 3;           // stored row (channel) / matrix this lane addresses
      const int hv = RAG ? min(max(__ldg(valid + n), 0), H) : H;      // RAG only
#pragma unroll 1
      for (int rd = 0; rd < ROUNDS; ++rd) {
        uint32_t q[4][4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int gi = warp + 8 * (rd * 4 + u);
#pragma unroll
          for (int mi = 0; mi < 4; ++mi) {
            const int m = 4 * gi + mi;
            const int r = m / WB, wb = m - r * WB;
            const int h = h0 - 3 + r, w = wb * 8 + px;
            const bool ok = m < NM && (RAG ? (unsigned)h < (unsigned)hv : (h >= 0 && h < H)) && w < W;
            q[u][mi] = ok ? ldg_nc_u32(xin + ((size_t)h * W + w) * C) : 0u;
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int gi = warp + 8 * (rd * 4 + u);
          if (gi < NG) {                                  // warp-uniform
            const int m = 4 * gi + smi;
            const int r = m / WB, wb = m - r * WB;
            const uint32_t dst = m < NM ? s_base + OFF_A + sj * A_STRIDE + r * 128 + ((wb ^ ((sj + r) & 7)) << 4)
                                        : s_base + OFF_DUMMY + lane * 16;
            stmatrix_x4_trans(dst, q[u][0], q[u][1], q[u][2], q[u][3]);
          }
        }
      }
    }
    ptx::fence_proxy_async_smem();
    __syncthreads();

#pragma unroll 1
    for (int half = 0; half < NHALF; ++half) {
      if (warp == 0) {
        // ---- MMA issuer --------------------------------------------------------------------------------------------
        if (ptx::elect_one()) {
          constexpr uint32_t idesc = ptx::umma_idesc_bf16(64, 32);
          uint32_t my_bc = bc;
#pragma unroll 1
          for (int c = 0; c < CG; ++c, ++my_bc) {
            const int slot = my_bc & 1;
            ptx::mbar_wait(&band_full[slot], (my_bc >> 1) & 1);
            ptx::tc_fence_after();
            const uint64_t da = ptx::umma_desc_sw128_kmajor(s_base + OFF_A + c * A_STRIDE + half * 48);
            const uint64_t db = ptx::umma_desc_sw64_kmajor(s_base + OFF_BAND + slot * BAND);
            const uint32_t d = tmem + c * 32;
#pragma unroll
            for (int dy = 0; dy < 7; ++dy)
#pragma unroll
              for (int ks = 0; ks < 2; ++ks)
                ptx::umma_bf16(d, da + dy * 8 + 2 * ks, db + dy * (BAND_TILE / 16) + 2 * ks, idesc, (dy | ks) ? 1u : 0u);
            ptx::umma_commit(&band_empty[slot]);
          }
          ptx::umma_commit(d_full);
        }
        __syncwarp();
      } else {
        // ---- band builders ------------------------------------------------------------------------------------------
        uint32_t my_bc = bc;
#pragma unroll 1
        for (int c = 0; c < CG; ++c, ++my_bc) {
          const int slot = my_bc & 1;
          ptx::mbar_wait(&band_empty[slot], ((my_bc >> 1) & 1) ^ 1);
          if (b_ok) {
            uint8_t* dst = smem + OFF_BAND + slot * BAND + b_off;
            const uint16_t* tp = taps_s + c * 49 + bdx;
#pragma unroll
            for (int dy = 0; dy < 7; ++dy) *reinterpret_cast<uint16_t*>(dst + dy * BAND_TILE) = tp[dy * 7];
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&band_full[slot]);
        }
      }
      bc += CG;
      // ---- write-out: TMEM -> +bias -> bf16 -> NHWC ---------------------------------------------------------------------
      ptx::mbar_wait(d_full, dphase);
      dphase ^= 1;
      ptx::tc_fence_after();
      {
        const int q4 = warp & 3, side = warp >> 2;          // TMEM lane quadrant; which 16 accumulator columns
        const int m = q4 * 16 + lane;                        // M = 64: row m sits in lane (m / 16) * 32 + m % 16
        const int h = h0 + m;
        const bool row_ok = lane < 16 && m < TR && h < H;
        const uint32_t ta = tmem + (static_cast<uint32_t>(q4 * 32) << 16);
        float bs[CG];
#pragma unroll
        for (int c = 0; c < CG; ++c) bs[c] = bias[c0 + c];
        bf16* vrow = v + (((size_t)n * H + (row_ok ? h : 0)) * W) * C + c0;
#pragma unroll
        for (int b = 0; b < 2; ++b) {
          const int col0 = side * 16 + b * 8;                // accumulator columns [col0, col0 + 8)
          uint32_t r[CG][8];
#pragma unroll
          for (int c = 0; c < CG; ++c) tmem_ld_32x32b_x8(ta + c * 32 + col0, r[c]);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int col = col0 + j;
            // left half: output column = col (valid below 28 resp. W); right half: output column = 24 + col, col >= 4
            const int w = half == 0 ? col : 24 + col;
            const bool ok = row_ok && (half == 0 ? col < (NHALF == 2 ? 28 : W) : col >= 4);
            if (ok) {
              uint4 o;
              o.x = Pair<bf16>::pack(__uint_as_float(r[0][j]) + bs[0], __uint_as_float(r[1][j]) + bs[1]);
              o.y = Pair<bf16>::pack(__uint_as_float(r[2][j]) + bs[2], __uint_as_float(r[3][j]) + bs[3]);
              o.z = Pair<bf16>::pack(__uint_as_float(r[4][j]) + bs[4], __uint_as_float(r[5][j]) + bs[5]);
              o.w = Pair<bf16>::pack(__uint_as_float(r[6][j]) + bs[6], __uint_as_float(r[7][j]) + bs[7]);
              *reinterpret_cast<uint4*>(vrow + (size_t)w * C) = o;
            }
          }
        }
      }
      ptx::tc_fence_before();
      __syncthreads();                  // accumulators drained (next half / unit overwrites them); A tiles free after the last half
      ptx::tc_fence_after();
    }
  }
  if (warp == 0) ptx::tmem_dealloc(tmem, 256);
}

// =====================================================================================================================
// v3 (group-planar only): ONE persistent CTA per SM that owns a FIXED 8-channel group.
// Group-planar activations: x and v are [C/8][Mp][8] (M = clips * H * W pixels, Mp = M rounded up to 128 = the plane
// stride; every 16-byte group of 8 channels is a plane).  With NHWC tensors a unit's 16-byte pieces sit 2 C bytes apart:
// each costs the LSU a 32-byte sector request and the staging / write-out phases of the kernel above ran at ~5 useful
// B/clk/SM (24 k + 8 k of a unit's 54 k cycles, in-kernel clock trace, commit 17b9d13; TMA gathers the same pieces at
// 14 B/clk/SM, tools/ubench/tma_gather.cu).  In the planar layout a unit's image rows are contiguous: fragment loads are
// full 128-byte lines and the results leave as contiguous runs.
//   * the 8 x 7 band matrices of its channels (112 KB) are built once and stay in shared memory: no per-channel band
//     build / hand-off in steady state (in-kernel clock traces of the kernel above, commit 17b9d13: ~1.0 k cycles per
//     channel against 0.34 k of MMA time, bands + MMA were 44 % of a unit);
//   * the work item is a (clip, 63-row tile, half row): its A tile holds only the 32-column K window of that half
//     (64-byte rows, SWIZZLE_64B, 36.5 KB for 8 channels), so TWO of them fit and the accumulators of two items fit the
//     512 TMEM columns -- loaders, the MMA thread and the write-out warps work on three different items at once:
//       warps 1-7   loaders: fragment loads (full 128-byte lines of the planar tensor) -> stmatrix.trans -> A[buf];
//                   ALL rows of an item are requested in one round (10 rows = 40 loads in flight per lane): with four
//                   warps and three dependent rounds per item the loaders were latency-bound (7.4 k cycles per item
//                   against 2.75 k of MMA time); an L2 prefetch of the next item's rows changed nothing (110.8 vs 110.2 us):
//                   the loaders are bound by their own instruction stream (40 loads + 10 stmatrix per lane and item)
//       warp  0     112 back-to-back tcgen05.mma (M64 N32 K16) per item -> D[buf]
//       warps 8-15  write-out: D[buf] -> + bias -> bf16 -> smem staging -> 448-byte contiguous runs of the planar output
// =====================================================================================================================
namespace v3 {
constexpr int A_CH = 73 * 64;                  // bytes between the channels' A tiles (73 rows of 64 B; 73 == 1 mod 8)
constexpr int A_BUF = CG * A_CH;               // 37376
constexpr int OFF_BANDS = 0;                   // [8 ch][7 dy][32 x 64 B]
constexpr int OFF_A = CG * BAND;               // 114688
constexpr int OFF_STG = OFF_A + 2 * A_BUF;     // write-out staging [63][28 x 16 B]
constexpr int STG_PITCH = 28 * 16 + 16;        // 464 B: 16 rows written at once land in 16 different bank groups
constexpr int OFF_MISC = OFF_STG + TR * STG_PITCH + 64;   // bias[8]
constexpr int OFF_BAR = OFF_MISC + 64;
constexpr int SMEM_BYTES = OFF_BAR + 128 + 1024;
constexpr int THREADS = 512;
constexpr int NLOAD = 7;                       // loader warps
static_assert(OFF_A % 1024 == 0 && A_BUF % 512 == 0, "swizzle atoms");
static_assert(SMEM_BYTES <= 227 * 1024, "smem budget");

// RAG: as in dwconv_tc_kernel; a paired item (W = 14) bounds each of its two clips by its own valid[] entry.
template <int W, bool RAG = false>
__global__ void __launch_bounds__(THREADS, 1)
    dwconv_tc3_kernel(const bf16* __restrict__ x, const bf16* __restrict__ taps /*[49][C]*/, const float* __restrict__ bias,
                      bf16* __restrict__ v, int n_clips, int H, int C, const int32_t* __restrict__ valid) {
  constexpr int NHALF = W > 32 ? 2 : 1;
  constexpr int HW = NHALF == 2 ? 28 : W;
  // W = 14: an item takes the rows of TWO clips side by side in one 32-column K window -- clip A in columns 0..13, three
  // zero columns (the conv's own padding, so the band couples nothing across them), clip B in columns 17..30 -- because
  // an item's cost is mostly fixed hand-offs (a 14-wide item alone took as long as a 28-wide one: 56 us per layer)
  constexpr bool PAIR = W == 14;
  constexpr int KS = 2;                         // K steps per (channel, dy)
  constexpr int NMI = 4;                        // 8-pixel blocks per A row
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t s_base = ptx::smem_u32(smem);
  float* sbias = reinterpret_cast<float*>(smem + OFF_MISC);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* a_full = bars;          // [2] loaders -> MMA
  uint64_t* a_empty = bars + 2;     // [2] MMA (commit) -> loaders
  uint64_t* d_full = bars + 4;      // [2] MMA (commit) -> write-out
  uint64_t* d_empty = bars + 6;     // [2] write-out -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int G = C / CG;
  const int g = blockIdx.x % G, rank = blockIdx.x / G;
  const int ng = ((int)gridDim.x - g + G - 1) / G;            // CTAs that own this channel group
  const int tiles = (H + TR - 1) / TR;
  const int items = (PAIR ? (n_clips + 1) / 2 : n_clips) * tiles * NHALF;
  const int c0 = g * CG;
  const size_t mtot = ((size_t)n_clips * H * W + 127) / 128 * 128;   // plane stride: rows rounded up to 128

  // ---- once per CTA: zero everything the MMAs may read, then the band diagonals of the 8 channels ----------------------
  for (int i = tid; i < OFF_STG / 16; i += THREADS) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  if (tid < CG) sbias[tid] = bias[c0 + tid];
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&a_full[s], NLOAD);
      ptx::mbar_init(&a_empty[s], 1);
      ptx::mbar_init(&d_full[s], 1);
      ptx::mbar_init(&d_empty[s], 8);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 0) {
    ptx::tmem_alloc(tmem_slot, 512);
    ptx::tmem_relinquish();
  }
  // the 8 channels' 49 taps first (49 coalesced 16-byte loads into the still unused staging area): building the bands
  // straight from global memory cost ~25 dependent L2 round trips per thread, 8 us of a 40 us stage-2 launch
  uint16_t* taps_s = reinterpret_cast<uint16_t*>(smem + OFF_STG);          // [49][8]
  if (tid < 49) reinterpret_cast<uint4*>(taps_s)[tid] = __ldg(reinterpret_cast<const uint4*>(taps + (size_t)tid * C + c0));
  __syncthreads();
  for (int i = tid; i < CG * 49 * 32; i += THREADS) {          // (channel, tap, n): T[n][k = n + dx - 3] = tap[dy][dx]
    const int n = i & 31, tap = (i >> 5) % 49, c = i / (49 * 32);
    const int dy = tap / 7, dx = tap - dy * 7, k = n + dx - 3;
    if (k >= 0 && k < 32)
      *reinterpret_cast<uint16_t*>(smem + OFF_BANDS + (c * 7 + dy) * BAND_TILE + n * 64 +
                                   ((((k >> 3) ^ ((n >> 1) & 3)) << 4) + ((k & 7) << 1))) = taps_s[tap * 8 + c];
  }
  ptx::fence_proxy_async_smem();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  pdl_trigger();       // TMEM allocated, bands built: everything above read only this layer's taps and bias, so under
  pdl_wait();          // programmatic dependent launch it overlaps the tail of the kernel that produces x

  if (warp == 0) {
    // ===================== MMA issuer ==================================================================================
    if (ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::umma_idesc_bf16(64, 32);
      uint32_t it = 0;
      for (int item = rank; item < items; item += ng, ++it) {
        const int buf = it & 1;
        const uint32_t par = (it >> 1) & 1;
        ptx::mbar_wait(&a_full[buf], par);
        ptx::mbar_wait(&d_empty[buf], par ^ 1);
        ptx::tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < CG; ++c) {
          const uint64_t da = ptx::umma_desc_sw64_kmajor(s_base + OFF_A + buf * A_BUF + c * A_CH);
          const uint64_t db = ptx::umma_desc_sw64_kmajor(s_base + OFF_BANDS + c * BAND);
          const uint32_t d = tmem + buf * 256 + c * 32;
#pragma unroll
          for (int dy = 0; dy < 7; ++dy)
#pragma unroll
            for (int ks = 0; ks < KS; ++ks)
              ptx::umma_bf16(d, da + dy * 4 + 2 * ks, db + dy * (BAND_TILE / 16) + 2 * ks, idesc, (dy | ks) ? 1u : 0u);
        }
        ptx::umma_commit(&a_empty[buf]);
        ptx::umma_commit(&d_full[buf]);
      }
    }
  } else if (warp >= 1 && warp <= NLOAD) {
    // ===================== loaders ==========================================================================================
    const int lw = warp - 1;
    const int px = lane >> 2;                           // pixel of the fragment this lane loads
    const int sj = lane & 7, smi = lane >> 3;           // stored row (channel) / matrix (8-pixel block) this lane addresses
    const bf16* xg = x + (size_t)g * mtot * 8 + 2 * (lane & 3);
    uint32_t it = 0;
    for (int item = rank; item < items; item += ng, ++it) {
      const int half = item % NHALF, t = (item / NHALF) % tiles, n = (item / (NHALF * tiles)) * (PAIR ? 2 : 1);
      const int h0 = t * TR, kw0 = half ? 24 : 0;
      const int buf = it & 1;
      ptx::mbar_wait(&a_empty[buf], ((it >> 1) & 1) ^ 1);
      const bf16* xin = xg + ((size_t)n * H * W + kw0) * 8;
      const bool b_ok = PAIR && n + 1 < n_clips;        // the pair's second clip exists
      const int hv_a = RAG ? min(max(__ldg(valid + n), 0), H) : H;
      const int hv_b = RAG && b_ok ? min(max(__ldg(valid + n + 1), 0), H) : H;
      const uint32_t abuf = s_base + OFF_A + buf * A_BUF;
      constexpr int RPR = (AR + NLOAD - 1) / NLOAD;     // rows per warp: all requested at once
#pragma unroll 1
      for (int r0 = lw; r0 < AR; r0 += NLOAD * RPR) {
        uint32_t q[RPR][4];
#pragma unroll
        for (int u = 0; u < RPR; ++u) {
          const int r = r0 + NLOAD * u, h = h0 - 3 + r;
          const bool row_ok = r < AR && h >= 0 && h < hv_a;
#pragma unroll
          for (int mi = 0; mi < 4; ++mi) {
            const int col = kw0 + mi * 8 + px;
            if (PAIR) {
              const int ca = mi * 8 + px;               // A column: 0..13 clip A, 17..30 clip B
              const bool in_a = ca < 14, in_b = ca >= 17 && ca < 31 && b_ok;
              const size_t off = in_a ? ((size_t)h * W + ca) : ((size_t)(H + h) * W + ca - 17);
              if (RAG) {                                // row_ok bounds clip A only
                const bool rb = r < AR && h >= 0 && h < hv_b;
                q[u][mi] = ((in_a && row_ok) || (in_b && rb)) ? ldg_nc_u32(xin + off * 8) : 0u;
              } else {
                q[u][mi] = (row_ok && (in_a || in_b)) ? ldg_nc_u32(xin + off * 8) : 0u;
              }
            } else {
              q[u][mi] = (mi < NMI && row_ok && col < W) ? ldg_nc_u32(xin + ((size_t)h * W + mi * 8 + px) * 8) : 0u;
            }
          }
        }
#pragma unroll
        for (int u = 0; u < RPR; ++u) {
          const int r = r0 + NLOAD * u;
          if (r < AR)                                   // warp-uniform
            stmatrix_x4_trans(abuf + sj * A_CH + r * 64 + ((smi ^ (((sj * 73 + r) >> 1) & 3)) << 4), q[u][0], q[u][1],
                              q[u][2], q[u][3]);
        }
      }
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&a_full[buf]);
    }
  } else if (warp >= 8) {
    // ===================== write-out =========================================================================================
    // An M = 64 accumulator occupies lanes 0..15 of each 32-lane TMEM quadrant, so the 32x32b load shape would move
    // (and the 16 idle lanes of every warp would wait for) twice the data; 16x256b reads exactly those 16 lanes x 8
    // columns and hands thread t the accumulator-fragment elements (row t/4, columns 2(t%4), 2(t%4)+1) and (row t/4 + 8,
    // same columns): every lane packs 4 pixels x 8 channels.  (First version: 32x32b.x8, write-out 4.9 k cycles per
    // item against 2.9 k of MMA time -- the slowest role.)
    const int ew = warp - 8;
    const int q4 = ew & 3, side = ew >> 2;              // TMEM lane quadrant (== warp % 4); which 16 accumulator columns
    const uint32_t ta = tmem + (static_cast<uint32_t>(q4 * 32) << 16);
    const int etid = tid - 256;
    const int m_a = q4 * 16 + (lane >> 2), m_b = m_a + 8;       // the two rows this lane holds
    float bs[CG];
#pragma unroll
    for (int c = 0; c < CG; ++c) bs[c] = sbias[c];
    uint32_t it = 0;
    for (int item = rank; item < items; item += ng, ++it) {
      const int half = item % NHALF, t = (item / NHALF) % tiles, n = (item / (NHALF * tiles)) * (PAIR ? 2 : 1);
      const int h0 = t * TR;
      const int buf = it & 1;
      ptx::mbar_wait(&d_full[buf], (it >> 1) & 1);
      ptx::tc_fence_after();
      uint32_t r[2][CG][4];
#pragma unroll
      for (int b = 0; b < 2; ++b)
#pragma unroll
        for (int c = 0; c < CG; ++c)
          asm volatile("tcgen05.ld.sync.aligned.16x256b.x1.b32 {%0, %1, %2, %3}, [%4];"
                       : "=r"(r[b][c][0]), "=r"(r[b][c][1]), "=r"(r[b][c][2]), "=r"(r[b][c][3])
                       : "r"(ta + buf * 256 + c * 32 + side * 16 + b * 8)
                       : "memory");
      // the previous item's bulk copies must have finished READING the staging rows before they are rewritten
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      asm volatile("bar.sync 1, 256;" ::: "memory");
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&d_empty[buf]);   // all of this warp's TMEM reads of the item have landed
#pragma unroll
      for (int b = 0; b < 2; ++b) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int mm = (e & 2) ? m_b : m_a;
          const int col = side * 16 + b * 8 + 2 * (lane & 3) + (e & 1);
          // staging slot of this accumulator column: pixel of the half row; PAIR: clip A 0..13, clip B 14..27
          const int slot = PAIR ? (col < 14 ? col : col - 3) : (half == 0 ? col : col - 4);
          const bool ok = mm < TR && h0 + mm < H &&
                          (PAIR ? (col < 14 || (col >= 17 && col < 31)) : (half == 0 ? col < HW : col >= 4));
          if (ok) {
            uint4 o;
            o.x = Pair<bf16>::pack(__uint_as_float(r[b][0][e]) + bs[0], __uint_as_float(r[b][1][e]) + bs[1]);
            o.y = Pair<bf16>::pack(__uint_as_float(r[b][2][e]) + bs[2], __uint_as_float(r[b][3][e]) + bs[3]);
            o.z = Pair<bf16>::pack(__uint_as_float(r[b][4][e]) + bs[4], __uint_as_float(r[b][5][e]) + bs[5]);
            o.w = Pair<bf16>::pack(__uint_as_float(r[b][6][e]) + bs[6], __uint_as_float(r[b][7][e]) + bs[7]);
            *reinterpret_cast<uint4*>(smem + OFF_STG + mm * STG_PITCH + slot * 16) = o;
          }
        }
      }
      ptx::fence_proxy_async_smem();                    // staging (generic writes) -> bulk-copy engine (async proxy)
      asm volatile("bar.sync 1, 256;" ::: "memory");    // staging complete (write-out warps only)
      const int rows = min(TR, H - h0);
      if (etid < rows) {                                // one bulk copy per image row: HW x 16 contiguous bytes
        bf16* vg = v + ((size_t)g * mtot + ((size_t)n * H + h0 + etid) * W + (half == 0 ? 0 : 28)) * 8;
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(vg),
                     "r"(s_base + OFF_STG + etid * STG_PITCH), "n"(HW * 16)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      } else if (PAIR && etid >= 64 && etid - 64 < rows && n + 1 < n_clips) {     // the pair's second clip
        const int row = etid - 64;
        bf16* vg = v + ((size_t)g * mtot + ((size_t)(n + 1) * H + h0 + row) * W) * 8;
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(vg),
                     "r"(s_base + OFF_STG + row * STG_PITCH + HW * 16), "n"(HW * 16)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");    // all stores complete before the CTA exits
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem, 512);
  }
}

template <int W, bool RAG>
static int launch(const void* x, const void* taps, const float* bias, void* v, int B, int H, int C, const int32_t* valid,
                  cudaStream_t st) {
  auto kern = dwconv_tc3_kernel<W, RAG>;
  ACX_SET_MAX_SMEM(kern, SMEM_BYTES);
  const int G = C / CG;
  const long long work = (long long)G * (W == 14 ? (B + 1) / 2 : B) * ceil_div(H, TR) * (W > 32 ? 2 : 1);
  const int sms = sm_count();
  const int grid = work < sms ? (int)work : sms;       // >= G whenever there is at least one item per group
  ACX_CUDA(launch_pdl(kern, dim3(grid), dim3(THREADS), SMEM_BYTES, st, 1, PDL_DWTC, reinterpret_cast<const bf16*>(x),
                      reinterpret_cast<const bf16*>(taps), bias, reinterpret_cast<bf16*>(v), B, H, C, valid));
  return ACX_OK;
}
}  // namespace v3

template <int W, bool RAG>
static int launch(const void* x, const void* taps, const float* bias, void* v, int B, int H, int C, const int32_t* valid,
                  cudaStream_t st) {
  auto kern = dwconv_tc_kernel<W, RAG>;
  ACX_SET_MAX_SMEM(kern, SMEM_BYTES);
  const int units = B * ceil_div(H, TR) * (C / CG);
  const int grid = units < 2 * sm_count() ? units : 2 * sm_count();
  kern<<<grid, THREADS, SMEM_BYTES, st>>>(reinterpret_cast<const bf16*>(x), reinterpret_cast<const bf16*>(taps), bias,
                                          reinterpret_cast<bf16*>(v), B, H, C, valid);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

// ---- channels-last LayerNorm over rows of C bf16 values (reference convnext.py:78, eps 1e-6), in place capable ----------
// C / 24 lanes per row, three 16-byte vectors per lane (the ln_patchify scheme): every warp instruction moves whole
// rows, statistics are two-pass in registers (mean, then centred sum of squares) with log2(C/24) shuffles.
template <int C>
__global__ void __launch_bounds__(256, 4)
    layernorm_rows_kernel(const bf16* __restrict__ in, const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                          bf16* __restrict__ out, long long M) {
  constexpr int CH = 24, LPP = C / CH, NPIX = 2;
  static_assert(C % CH == 0 && (LPP & (LPP - 1)) == 0 && LPP <= 32, "lane split");
  const int lig = threadIdx.x % LPP;
  const long long grp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / LPP;
  const float* gp = ln_w + lig * CH;
  const float* bp = ln_b + lig * CH;
  float val[NPIX][CH];
  bool ok[NPIX];
#pragma unroll
  for (int q = 0; q < NPIX; ++q) {
    const long long row = grp * NPIX + q;
    ok[q] = row < M;
    const bf16* src = in + (ok[q] ? row : 0) * C + lig * CH;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const uint4 raw = __ldg(reinterpret_cast<const uint4*>(src) + j);
      float2 f;
      f = Pair<bf16>::unpack(raw.x); val[q][8 * j + 0] = f.x; val[q][8 * j + 1] = f.y;
      f = Pair<bf16>::unpack(raw.y); val[q][8 * j + 2] = f.x; val[q][8 * j + 3] = f.y;
      f = Pair<bf16>::unpack(raw.z); val[q][8 * j + 4] = f.x; val[q][8 * j + 5] = f.y;
      f = Pair<bf16>::unpack(raw.w); val[q][8 * j + 6] = f.x; val[q][8 * j + 7] = f.y;
    }
  }
#pragma unroll
  for (int q = 0; q < NPIX; ++q) {
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < CH; ++j) sum += val[q][j];
#pragma unroll
    for (int o = LPP / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float mean = sum * (1.0f / C);
    float sq = 0.f;
#pragma unroll
    for (int j = 0; j < CH; ++j) {
      val[q][j] -= mean;
      sq = fmaf(val[q][j], val[q][j], sq);
    }
#pragma unroll
    for (int o = LPP / 2; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    const float rstd = rsqrtf(sq * (1.0f / C) + 1e-6f);
    if (ok[q]) {
      bf16* dst = out + (grp * NPIX + q) * C + lig * CH;
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const int k = 8 * j;
        const float4 g0 = __ldg(reinterpret_cast<const float4*>(gp + k)), g1 = __ldg(reinterpret_cast<const float4*>(gp + k + 4));
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(bp + k)), b1 = __ldg(reinterpret_cast<const float4*>(bp + k + 4));
        uint4 o4;
        o4.x = Pair<bf16>::pack(val[q][k + 0] * rstd * g0.x + b0.x, val[q][k + 1] * rstd * g0.y + b0.y);
        o4.y = Pair<bf16>::pack(val[q][k + 2] * rstd * g0.z + b0.z, val[q][k + 3] * rstd * g0.w + b0.w);
        o4.z = Pair<bf16>::pack(val[q][k + 4] * rstd * g1.x + b1.x, val[q][k + 5] * rstd * g1.y + b1.y);
        o4.w = Pair<bf16>::pack(val[q][k + 6] * rstd * g1.z + b1.z, val[q][k + 7] * rstd * g1.w + b1.w);
        reinterpret_cast<uint4*>(dst)[j] = o4;
      }
    }
  }
}

template <int C>
static int launch_ln(const void* in, const float* ln_w, const float* ln_b, void* out, long long M, cudaStream_t st) {
  constexpr int LPP = C / 24, NPIX = 2;
  const long long lanes = (M + NPIX - 1) / NPIX * LPP;
  const long long blocks = (lanes + 255) / 256;
  layernorm_rows_kernel<C><<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const bf16*>(in), ln_w, ln_b,
                                                             reinterpret_cast<bf16*>(out), M);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

}  // namespace dwtc
}  // namespace acx

using namespace acx;

template <bool RAG>
static int dwconv_tc_impl(const void* x, const void* w, const float* bias, void* v, int B, int H, int W, int C,
                          const int32_t* valid, void* stream) {
  ACX_CHECK(x && w && bias && v, ACX_ERR_ARG, "dwconv_tc: null pointer");
  ACX_CHECK(B > 0 && H > 0, ACX_ERR_ARG, "dwconv_tc: B and H must be positive");
  ACX_CHECK(C % 8 == 0 && C > 0, ACX_ERR_ARG, "dwconv_tc: C must be a positive multiple of 8 (got %d)", C);
  ACX_CHECK(x != v, ACX_ERR_ARG, "dwconv_tc: out of place only (neighbouring units read the input halo)");
  ACX_CHECK(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(v)) & 15) == 0, ACX_ERR_ARG,
            "dwconv_tc: x and v must be 16-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  switch (W) {
    case 56: return dwtc::launch<56, RAG>(x, w, bias, v, B, H, C, valid, st);
    case 28: return dwtc::launch<28, RAG>(x, w, bias, v, B, H, C, valid, st);
    case 14: return dwtc::launch<14, RAG>(x, w, bias, v, B, H, C, valid, st);
    case 7: return dwtc::launch<7, RAG>(x, w, bias, v, B, H, C, valid, st);
    default:
      set_error("dwconv_tc: W=%d not supported (the ConvNeXt stages are 56 / 28 / 14 / 7 wide)", W);
      return ACX_ERR_UNSUPPORTED;
  }
}

extern "C" int acx_dwconv_tc(const void* x, const void* w, const float* bias, void* v, int B, int H, int W, int C,
                             void* stream) {
  return dwconv_tc_impl<false>(x, w, bias, v, B, H, W, C, nullptr, stream);
}

extern "C" int acx_dwconv_tc_ragged(const void* x, const void* w, const float* bias, void* v, int B, int H, int W, int C,
                                    const int32_t* valid, void* stream) {
  ACX_CHECK(valid, ACX_ERR_ARG, "dwconv_tc_ragged: null valid-length array");
  return dwconv_tc_impl<true>(x, w, bias, v, B, H, W, C, valid, stream);
}

// Same on group-planar activations: x, v = [C/8][B*H*W][8] bf16.
template <bool RAG>
static int dwconv_tc_gp_impl(const void* x, const void* w, const float* bias, void* v, int B, int H, int W, int C,
                             const int32_t* valid, void* stream) {
  ACX_CHECK(x && w && bias && v, ACX_ERR_ARG, "dwconv_tc_gp: null pointer");
  ACX_CHECK(B > 0 && H > 0, ACX_ERR_ARG, "dwconv_tc_gp: B and H must be positive");
  ACX_CHECK(C % 8 == 0 && C > 0, ACX_ERR_ARG, "dwconv_tc_gp: C must be a positive multiple of 8 (got %d)", C);
  ACX_CHECK(x != v, ACX_ERR_ARG, "dwconv_tc_gp: out of place only (neighbouring units read the input halo)");
  ACX_CHECK(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(w)) & 15) == 0,
            ACX_ERR_ARG, "dwconv_tc_gp: x, v and w must be 16-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  switch (W) {
    case 56: return dwtc::v3::launch<56, RAG>(x, w, bias, v, B, H, C, valid, st);
    case 28: return dwtc::v3::launch<28, RAG>(x, w, bias, v, B, H, C, valid, st);
    case 14: return dwtc::v3::launch<14, RAG>(x, w, bias, v, B, H, C, valid, st);
    default:
      set_error("dwconv_tc_gp: W=%d not supported (stages 0 - 2: 56 / 28 / 14)", W);
      return ACX_ERR_UNSUPPORTED;
  }
}

extern "C" int acx_dwconv_tc_gp(const void* x, const void* w, const float* bias, void* v, int B, int H, int W, int C,
                                void* stream) {
  return dwconv_tc_gp_impl<false>(x, w, bias, v, B, H, W, C, nullptr, stream);
}

extern "C" int acx_dwconv_tc_gp_ragged(const void* x, const void* w, const float* bias, void* v, int B, int H, int W, int C,
                                       const int32_t* valid, void* stream) {
  ACX_CHECK(valid, ACX_ERR_ARG, "dwconv_tc_gp_ragged: null valid-length array");
  return dwconv_tc_gp_impl<true>(x, w, bias, v, B, H, W, C, valid, stream);
}

// ---- (M, C) row-major <-> group-planar [C/8][M][8] ----------------------------------------------------------------------
// One block moves 64 rows: 16-byte pieces are read along the source's contiguous direction and written along the
// destination's (both sides whole lines) through a padded smem tile.
namespace acx {
namespace dwtc {
__global__ void __launch_bounds__(256) gp_transpose_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, long long M,
                                                           int G, int to_gp) {
  extern __shared__ uint4 tile[];                 // [64 rows][G + 1]
  const long long r0 = (long long)blockIdx.x * 64;
  const int rows = (int)min((long long)64, M - r0);
  const int pitch = G + 1;
  const long long Mp = (M + 127) / 128 * 128;     // plane stride of the planar side
  if (to_gp) {
    for (int i = threadIdx.x; i < rows * G; i += 256) {          // row-major source: consecutive i = consecutive pieces of a row
      const int r = i / G, gq = i - r * G;
      tile[r * pitch + gq] = in[(r0 + r) * G + gq];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < rows * G; i += 256) {          // planar destination: consecutive i = consecutive rows of a plane
      const int gq = i / rows, r = i - gq * rows;
      out[(long long)gq * Mp + r0 + r] = tile[r * pitch + gq];
    }
  } else {
    for (int i = threadIdx.x; i < rows * G; i += 256) {
      const int gq = i / rows, r = i - gq * rows;
      tile[r * pitch + gq] = in[(long long)gq * Mp + r0 + r];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < rows * G; i += 256) {
      const int r = i / G, gq = i - r * G;
      out[(r0 + r) * G + gq] = tile[r * pitch + gq];
    }
  }
}
}  // namespace dwtc
}  // namespace acx

// Per-row LayerNorm statistics of a group-planar tensor [C/8][Mp][8] bf16: stats[row] = (rstd, -mean * rstd), eps 1e-6.
// For the stages whose MLP is the N-tiled generic GEMM: every N tile's GELU epilogue needs the row's statistics and
// none of them owns the row, so they are computed once here (one pass over v: thread = row, loads coalesced per plane).
namespace acx {
namespace dwtc {
__global__ void __launch_bounds__(128) gp_row_stats_kernel(const uint4* __restrict__ v, float2* __restrict__ stats,
                                                           long long M, int G) {
  pdl_trigger();
  pdl_wait();
  const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= M) return;
  const long long Mp = (M + 127) / 128 * 128;
  const float inv_c = 1.0f / (8.0f * G);
  const uint4 first = __ldg(v + row);
  const float shift = __uint_as_float(first.x << 16);
  const float2 sh2 = make_float2(-shift, -shift);
  float2 s = make_float2(0.f, 0.f), q = make_float2(0.f, 0.f);
  for (int g0 = 0; g0 < G; g0 += 12) {            // 12 independent 16-byte loads in flight per thread
    uint4 u[12];
#pragma unroll
    for (int j = 0; j < 12; ++j) u[j] = g0 + j < G ? __ldg(v + (long long)(g0 + j) * Mp + row) : make_uint4(0, 0, 0, 0);
#pragma unroll
    for (int j = 0; j < 12; ++j) {
      if (g0 + j < G) {
        const uint32_t w[4] = {u[j].x, u[j].y, u[j].z, u[j].w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 d = __fadd2_rn(Pair<bf16>::unpack(w[k]), sh2);
          s = __fadd2_rn(s, d);
          q = __ffma2_rn(d, d, q);
        }
      }
    }
  }
  const float md = (s.x + s.y) * inv_c;
  const float var = fmaxf((q.x + q.y) * inv_c - md * md, 0.f);
  const float rstd = rsqrtf(var + 1e-6f);
  stats[row] = make_float2(rstd, -(md + shift) * rstd);
}
}  // namespace dwtc
}  // namespace acx

extern "C" int acx_gp_row_stats(const void* v, float* stats, long long M, int C, void* stream) {
  ACX_CHECK(v && stats, ACX_ERR_ARG, "gp_row_stats: null pointer");
  ACX_CHECK(M > 0 && C > 0 && C % 8 == 0, ACX_ERR_ARG, "gp_row_stats: bad shape M=%lld C=%d", M, C);
  ACX_CUDA(launch_pdl(dwtc::gp_row_stats_kernel, dim3((unsigned)((M + 127) / 128)), dim3(128), 0, reinterpret_cast<cudaStream_t>(stream),
                      1, PDL_STATS, reinterpret_cast<const uint4*>(v), reinterpret_cast<float2*>(stats), M, C / 8));
  return ACX_OK;
}

extern "C" int acx_gp_transpose(const void* in, void* out, long long M, int C, int to_gp, void* stream) {
  ACX_CHECK(in && out && in != out, ACX_ERR_ARG, "gp_transpose: null or aliased pointers");
  ACX_CHECK(M > 0 && C > 0 && C % 8 == 0 && C <= 768, ACX_ERR_ARG, "gp_transpose: bad shape M=%lld C=%d", M, C);
  ACX_CHECK(((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15) == 0, ACX_ERR_ARG,
            "gp_transpose: 16-byte alignment");
  const int G = C / 8;
  const size_t smem = (size_t)64 * (G + 1) * 16;
  auto kern = dwtc::gp_transpose_kernel;
  ACX_SET_MAX_SMEM(kern, 64 * (768 / 8 + 1) * 16);       // the attribute is set once per device: size it for the widest C
  kern<<<(unsigned)((M + 63) / 64), 256, smem, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const uint4*>(in), reinterpret_cast<uint4*>(out), M, G, to_gp);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

extern "C" int acx_layernorm_rows(const void* in, const float* ln_w, const float* ln_b, void* out, long long M, int C,
                                  void* stream) {
  ACX_CHECK(in && ln_w && ln_b && out, ACX_ERR_ARG, "layernorm_rows: null pointer");
  ACX_CHECK(M > 0, ACX_ERR_ARG, "layernorm_rows: M must be positive");
  ACX_CHECK(((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15) == 0, ACX_ERR_ARG,
            "layernorm_rows: in and out must be 16-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  switch (C) {
    case 96: return dwtc::launch_ln<96>(in, ln_w, ln_b, out, M, st);
    case 192: return dwtc::launch_ln<192>(in, ln_w, ln_b, out, M, st);
    case 384: return dwtc::launch_ln<384>(in, ln_w, ln_b, out, M, st);
    case 768: return dwtc::launch_ln<768>(in, ln_w, ln_b, out, M, st);
    default:
      set_error("layernorm_rows: C=%d not supported (96 / 192 / 384 / 768)", C);
      return ACX_ERR_UNSUPPORTED;
  }
}
