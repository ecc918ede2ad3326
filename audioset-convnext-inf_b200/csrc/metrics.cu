// Tagging metrics: per-class exact integer counts (P, U2, S) behind average precision and ROC AUC (metrics.py is the
// host side and the reference).  Per chunk of classes: a pack kernel turns the row-major scores and labels into
// class-major 64-bit records and digit histograms, then one block per class radix-sorts its records by descending
// score and walks the tie groups from the top.
#include "common.cuh"

namespace acx {
namespace {

constexpr long long METRICS_MAX_N = 2147483647LL;   // row indices and counts fit 31 bits
constexpr int PK_THREADS = 1024;                    // pack: 32 warps
constexpr int PK_CLASSES = 32;                      // classes of one pack block (one per lane)
constexpr int PK_ROWS = 128;                        // rows of one pack tile (4 per warp)
constexpr int PK_HIST_STRIDE = 4 * 256 + 1;         // shared histogram words per class: the +1 spreads lanes over banks
constexpr int PK_SMEM = PK_CLASSES * PK_HIST_STRIDE * (int)sizeof(unsigned);
constexpr int MS_THREADS = 512, MS_WARPS = MS_THREADS / 32;
constexpr int MS_ITEMS = 4;                         // records per thread and tile
constexpr int MS_TILE = MS_THREADS * MS_ITEMS;

// Order key of a finite score: -0.0 is taken as +0.0, then the bits are made to compare as unsigned integers in the
// order of the values.
__device__ __forceinline__ unsigned order_key(float s) {
  unsigned u = __float_as_uint(s);
  if (u == 0x80000000u) u = 0u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// rec[c][r] = key(scores[r, c0 + c]) << 32 | (targets[r, c0 + c] != 0) for the block's 32 classes and its row range,
// written class-major to rec (kc, N); hist (kc, 4, 256) gains the counts of every byte of every key (pass p counts
// bits 8p .. 8p+7).  A tile is 128 rows x 32 classes: a warp reads 4 rows along the classes (coalesced), the tile is
// transposed in shared memory and a warp writes 128 rows of one class.
__global__ void __launch_bounds__(PK_THREADS)
    metrics_pack_kernel(const float* __restrict__ scores, const unsigned char* __restrict__ targets, long long N, int K,
                        int c0, int kc, long long rows_per_block, unsigned long long* __restrict__ rec,
                        unsigned* __restrict__ hist) {
  extern __shared__ unsigned sh_hist[];
  __shared__ unsigned long long tile[PK_ROWS][PK_CLASSES + 1];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cls0 = blockIdx.x * PK_CLASSES, nc = min(PK_CLASSES, kc - cls0);
  for (int i = tid; i < PK_CLASSES * PK_HIST_STRIDE; i += PK_THREADS) sh_hist[i] = 0u;
  __syncthreads();
  const long long r_begin = (long long)blockIdx.y * rows_per_block, r_end = min(N, r_begin + rows_per_block);
  for (long long r0 = r_begin; r0 < r_end; r0 += PK_ROWS) {
#pragma unroll
    for (int k = 0; k < PK_ROWS / 32; ++k) {
      const long long r = r0 + warp + 32 * k;
      if (r < r_end && lane < nc) {
        const long long e = r * K + c0 + cls0 + lane;
        const unsigned key = order_key(__ldg(scores + e));
        tile[warp + 32 * k][lane] = ((unsigned long long)key << 32) | (unsigned)(__ldg(targets + e) != 0);
        unsigned* h = sh_hist + lane * PK_HIST_STRIDE;
#pragma unroll
        for (int p = 0; p < 4; ++p) atomicAdd(h + p * 256 + ((key >> (8 * p)) & 255u), 1u);
      }
    }
    __syncthreads();
    if (warp < nc) {
      unsigned long long* dst = rec + (long long)(cls0 + warp) * N;
#pragma unroll
      for (int k = 0; k < PK_ROWS / 32; ++k) {
        const long long r = r0 + lane + 32 * k;
        if (r < r_end) dst[r] = tile[lane + 32 * k][warp];
      }
    }
    __syncthreads();
  }
  for (int i = tid; i < nc * 1024; i += PK_THREADS) {
    const unsigned v = sh_hist[(i >> 10) * PK_HIST_STRIDE + (i & 1023)];
    if (v) atomicAdd(hist + (long long)(cls0 + (i >> 10)) * 1024 + (i & 1023), v);
  }
}

// Exclusive scan of v over the block in thread order, under + (MAX false) or max (MAX true, identity 0); *total gets the
// block's total.  Every thread calls it.
template <bool MAX>
__device__ __forceinline__ unsigned long long block_exclusive(unsigned long long v, unsigned long long* tmp,
                                                              unsigned long long* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long incl = v;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, off);
    if (lane >= off) incl = MAX ? max(incl, t) : incl + t;
  }
  unsigned long long excl = __shfl_up_sync(0xffffffffu, incl, 1);
  if (lane == 0) excl = 0;
  __syncthreads();                                  // tmp may still be read by the previous call
  if (lane == 31) tmp[warp] = incl;
  __syncthreads();
  unsigned long long before = 0, all = 0;
#pragma unroll
  for (int w = 0; w < MS_WARPS; ++w) {
    const unsigned long long t = tmp[w];
    if (w < warp) before = MAX ? max(before, t) : before + t;
    all = MAX ? max(all, t) : all + t;
  }
  *total = all;
  return MAX ? max(before, excl) : before + excl;
}

// One block per class of the chunk.  rec_a holds the class's N records (from the pack); rec_b is the ping-pong buffer.
//
// Sort: a stable LSD radix sort by descending key, 8 bits a pass, passes whose histogram has a single non-empty bin
// skipped.  A pass walks the class tile by tile with running bucket offsets: each warp ranks its 128 records with
// __match_any_sync in index order, the per-warp counts are scanned across warps, the tile is staged in shared memory in
// digit order and written out in runs (consecutive records of one digit go to consecutive addresses).
//
// Scan: the sorted records are walked from the top, 2048 at a time, each thread owning 4 consecutive ones.  At record j
// (0-based, best first) pp = positives in [0, j]; a tie group [a, b) starts where the key differs from record j-1 and
// ends where it differs from record j+1.  A block max-scan of (a << 32 | positives before a) over the group starts
// gives every group end its start.  The group end adds n (2 PA + p) to U2 (p = positives in the group, n = negatives,
// PA = positives before it) and, when p > 0, floor(p TP 2^64 / C) (TP = positives up to its end, C = b) as three
// integer parts q, f1, f2 with S = q 2^64 + f1 2^32 + f2.  out[class] = (P, U2, S mod 2^64, S >> 64).
__global__ void __launch_bounds__(MS_THREADS)
    metrics_sort_scan_kernel(unsigned long long* rec_a, unsigned long long* rec_b, const unsigned* __restrict__ hist,
                             long long N, unsigned long long* __restrict__ out) {
  __shared__ unsigned warp_hist[MS_WARPS][256];
  __shared__ unsigned long long stage[MS_TILE];
  __shared__ unsigned bucket_off[256], tile_start[256], tile_cnt[256];
  __shared__ unsigned long long tmp[MS_WARPS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long cls = blockIdx.x;
  unsigned long long* src = rec_a + cls * N;
  unsigned long long* dst = rec_b + cls * N;
  const unsigned lanes_below = (1u << lane) - 1u;
  unsigned long long total;

  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 32 + 8 * pass;
    // slot 255 - digit: ascending slots are descending digits
    const unsigned h = tid < 256 ? __ldg(hist + cls * 1024 + pass * 256 + 255 - tid) : 0u;
    if (__syncthreads_or(tid < 256 && (long long)h == N)) continue;   // one bin holds every record: nothing moves
    const unsigned off = (unsigned)block_exclusive<false>(h, tmp, &total);
    if (tid < 256) bucket_off[tid] = off;
    for (long long t0 = 0; t0 < N; t0 += MS_TILE) {
      for (int i = tid; i < MS_WARPS * 256; i += MS_THREADS) (&warp_hist[0][0])[i] = 0u;
      __syncthreads();
      unsigned long long v[MS_ITEMS];
      unsigned slot[MS_ITEMS], rank[MS_ITEMS];
#pragma unroll
      for (int i = 0; i < MS_ITEMS; ++i) {
        const long long e = t0 + warp * (32 * MS_ITEMS) + i * 32 + lane;
        const bool valid = e < N;
        v[i] = valid ? src[e] : 0ull;
        slot[i] = valid ? 255u - (unsigned)((v[i] >> shift) & 255u) : 256u;   // 256: no record, a group of its own
        const unsigned peers = __match_any_sync(0xffffffffu, slot[i]);
        const unsigned before = valid ? warp_hist[warp][slot[i]] : 0u;
        __syncwarp();
        if (valid && (peers & lanes_below) == 0u) warp_hist[warp][slot[i]] = before + __popc(peers);
        __syncwarp();
        rank[i] = before + __popc(peers & lanes_below);
      }
      __syncthreads();
      unsigned cnt = 0;
      if (tid < 256) {
        for (int w = 0; w < MS_WARPS; ++w) {
          const unsigned t = warp_hist[w][tid];
          warp_hist[w][tid] = cnt;
          cnt += t;
        }
      }
      const unsigned start = (unsigned)block_exclusive<false>(cnt, tmp, &total);
      if (tid < 256) {
        tile_start[tid] = start;
        tile_cnt[tid] = cnt;
      }
      __syncthreads();
#pragma unroll
      for (int i = 0; i < MS_ITEMS; ++i)
        if (slot[i] < 256u) stage[tile_start[slot[i]] + warp_hist[warp][slot[i]] + rank[i]] = v[i];
      __syncthreads();
      const int n_tile = (int)min((long long)MS_TILE, N - t0);
      for (int j = tid; j < n_tile; j += MS_THREADS) {
        const unsigned long long x = stage[j];
        const unsigned s = 255u - (unsigned)((x >> shift) & 255u);
        dst[bucket_off[s] + (unsigned)j - tile_start[s]] = x;
      }
      __syncthreads();
      if (tid < 256) bucket_off[tid] += tile_cnt[tid];
    }
    unsigned long long* t = src;
    src = dst;
    dst = t;
    __syncthreads();
  }

  unsigned long long pp_carry = 0, start_carry = 0;
  unsigned long long u2 = 0, sq = 0, sf1 = 0, sf2 = 0;
  for (long long t0 = 0; t0 < N; t0 += MS_TILE) {
    const long long j0 = t0 + (long long)tid * MS_ITEMS;
    unsigned key[MS_ITEMS + 2], lab[MS_ITEMS];      // key[i + 1] is record j0 + i's; key[0] and key[5] its neighbours'
    unsigned lab_sum = 0;
#pragma unroll
    for (int i = 0; i < MS_ITEMS; ++i) {
      const unsigned long long x = j0 + i < N ? src[j0 + i] : 0ull;
      key[i + 1] = (unsigned)(x >> 32);
      lab[i] = (unsigned)(x & 1ull);
      lab_sum += lab[i];
    }
    key[0] = j0 > 0 && j0 < N ? (unsigned)(src[j0 - 1] >> 32) : 0u;
    key[MS_ITEMS + 1] = j0 + MS_ITEMS < N ? (unsigned)(src[j0 + MS_ITEMS] >> 32) : 0u;
    unsigned long long pp = pp_carry + block_exclusive<false>(lab_sum, tmp, &total);   // positives before j0
    pp_carry += total;
    unsigned long long st_local = 0;                 // (a << 32 | positives before a) of this thread's last start
    unsigned long long pp_run = pp;
#pragma unroll
    for (int i = 0; i < MS_ITEMS; ++i) {
      const long long j = j0 + i;
      if (j < N && (j == 0 || key[i] != key[i + 1])) st_local = ((unsigned long long)j << 32) | pp_run;
      pp_run += lab[i];
    }
    unsigned long long st = max(start_carry, block_exclusive<true>(st_local, tmp, &total));
    start_carry = max(start_carry, total);
#pragma unroll
    for (int i = 0; i < MS_ITEMS; ++i) {
      const long long j = j0 + i;
      if (j >= N) break;
      if (j == 0 || key[i] != key[i + 1]) st = ((unsigned long long)j << 32) | pp;
      pp += lab[i];
      if (j == N - 1 || key[i + 2] != key[i + 1]) {   // the end of the group [a, j + 1)
        const unsigned long long a = st >> 32, ppa = st & 0xffffffffull, b = (unsigned long long)j + 1;
        const unsigned long long p = pp - ppa, n = (b - a) - p;
        u2 += n * (2 * ppa + p);
        if (p) {
          const unsigned long long x = p * pp, q = x / b, r = x - q * b;
          const unsigned long long r32 = r << 32, f1 = r32 / b;
          sq += q;
          sf1 += f1;
          sf2 += ((r32 - f1 * b) << 32) / b;
        }
      }
    }
  }
  block_exclusive<false>(u2, tmp, &u2);
  block_exclusive<false>(sq, tmp, &sq);
  block_exclusive<false>(sf1, tmp, &sf1);
  block_exclusive<false>(sf2, tmp, &sf2);
  if (tid == 0) {
    const unsigned long long lo = (sf1 << 32) + sf2;
    const unsigned long long hi = sq + (sf1 >> 32) + (lo < (sf1 << 32) ? 1ull : 0ull);
    unsigned long long* o = out + cls * 4;
    o[0] = pp_carry;
    o[1] = u2;
    o[2] = lo;
    o[3] = hi;
  }
}

}  // namespace
}  // namespace acx

using namespace acx;

extern "C" {

int acx_tagging_metrics_workspace(long long N, int kc, long long* bytes) {
  ACX_CHECK(bytes, ACX_ERR_ARG, "tagging_metrics_workspace: null pointer");
  ACX_CHECK(N >= 1 && N <= METRICS_MAX_N && kc >= 1, ACX_ERR_ARG, "tagging_metrics_workspace: bad sizes N=%lld kc=%d",
            N, kc);
  *bytes = 2 * (long long)kc * N * (long long)sizeof(unsigned long long) + (long long)kc * 1024 * (long long)sizeof(unsigned);
  return ACX_OK;
}

int acx_tagging_metrics(const float* scores, long long N, int K, int c0, int kc, const unsigned char* targets,
                        void* workspace, unsigned long long* out, void* stream) {
  ACX_CHECK(scores && targets && workspace && out, ACX_ERR_ARG, "tagging_metrics: null pointer");
  ACX_CHECK(N >= 1 && N <= METRICS_MAX_N && K >= 1, ACX_ERR_ARG, "tagging_metrics: bad sizes N=%lld K=%d", N, K);
  ACX_CHECK(c0 >= 0 && kc >= 1 && c0 < K && kc <= K - c0, ACX_ERR_ARG,
            "tagging_metrics: classes [%d, %d + %d) outside [0, %d)", c0, c0, kc, K);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  unsigned long long* rec_a = static_cast<unsigned long long*>(workspace);
  unsigned long long* rec_b = rec_a + (long long)kc * N;
  unsigned* hist = reinterpret_cast<unsigned*>(rec_b + (long long)kc * N);
  ACX_CUDA(cudaMemsetAsync(hist, 0, (size_t)kc * 1024 * sizeof(unsigned), st));
  // about two pack blocks per SM (one fits at a time: its histograms take 128 KB of shared memory)
  const int groups = (kc + PK_CLASSES - 1) / PK_CLASSES;
  const long long tiles = (N + PK_ROWS - 1) / PK_ROWS;
  const long long splits = min(tiles, max(1LL, (2LL * sm_count() + groups - 1) / groups));
  const long long rows_per_block = (tiles + splits - 1) / splits * PK_ROWS;
  const dim3 grid((unsigned)groups, (unsigned)((N + rows_per_block - 1) / rows_per_block));
  ACX_SET_MAX_SMEM(metrics_pack_kernel, PK_SMEM);
  metrics_pack_kernel<<<grid, PK_THREADS, PK_SMEM, st>>>(scores, targets, N, K, c0, kc, rows_per_block, rec_a, hist);
  ACX_CUDA(cudaGetLastError());
  metrics_sort_scan_kernel<<<(unsigned)kc, MS_THREADS, 0, st>>>(rec_a, rec_b, hist, N, out);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

}  // extern "C"
