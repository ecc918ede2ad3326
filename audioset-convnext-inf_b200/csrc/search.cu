// Query by example: exact cosine scores in a fixed fp64 order and a per-query top k (search.py is the host side and the
// reference).
#include "common.cuh"

namespace acx {
namespace {

constexpr long long SEARCH_MAX_N = 2147483647LL;   // indices fit the low 32 bits of a hit's key
constexpr int SEARCH_MAX_K = 1024;                 // one hit per thread of the top-k block
constexpr int CS_BM = 64, CS_BN = 128, CS_BK = 16; // score tile: 64 queries x 128 keys, D staged 16 at a time
constexpr long long CS_MAX_Q = 65535LL * CS_BM;    // query tiles run on grid.y

// out[r] = sqrt(sum_i x[r, i]^2), the sum in fp64 in i order from 0.0 (each square of an fp32 value is exact in fp64, so
// fma(x, x, acc) rounds exactly like acc + x * x).  One thread per row.
__global__ void __launch_bounds__(256)
    row_norms_kernel(const float* __restrict__ x, long long rows, int d, double* __restrict__ out) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const float* p = x + r * d;
  double acc = 0.0;
  for (int i = 0; i < d; ++i) {
    const double v = (double)__ldg(p + i);
    acc = fma(v, v, acc);
  }
  out[r] = __dsqrt_rn(acc);
}

// scores[q, n] = float32(dot(q, n) / (qn[q] * kn[n])), dot the fp64 fma chain over i = 0 .. d-1 in order from 0.0, the
// product and quotient rounded once each in fp64 and the result rounded to nearest even; a NaN is stored as 0x7fc00000.
// Register-tiled SIMT DFMA GEMM: a block owns 64 queries x 128 keys, 128 threads own 8 x 8 outputs each (rows ty*4 + {0..3}
// and 32 + ty*4 + {0..3}, columns tx*4 + {0..3} and 64 + tx*4 + {0..3}, so every shared load is a broadcast-friendly
// LDS.128).  fp32 tiles of 16 dimensions are staged transposed in shared memory and widened in registers.  Only the
// dimensions that exist are chained: a zero-padded step would turn an accumulated -0.0 into +0.0.  Tensor cores are not
// used: neither tcgen05 nor DMMA promises this accumulation order.
__global__ void __launch_bounds__(128)
    cosine_scores_kernel(const float* __restrict__ qm, const double* __restrict__ qn, long long Q,
                         const float* __restrict__ km, const double* __restrict__ kn, long long N, int d,
                         float* __restrict__ scores) {
  __shared__ __align__(16) float As[CS_BK][CS_BM + 4];
  __shared__ __align__(16) float Bs[CS_BK][CS_BN + 4];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const long long q0 = (long long)blockIdx.y * CS_BM, n0 = (long long)blockIdx.x * CS_BN;
  double acc[8][8];
#pragma unroll
  for (int m = 0; m < 8; ++m)
#pragma unroll
    for (int n = 0; n < 8; ++n) acc[m][n] = 0.0;

  auto step = [&](int kk) {
    const float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
    const float4 a1 = *reinterpret_cast<const float4*>(&As[kk][32 + ty * 4]);
    const float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
    const float4 b1 = *reinterpret_cast<const float4*>(&Bs[kk][64 + tx * 4]);
    const double a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    const double b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int m = 0; m < 8; ++m)
#pragma unroll
      for (int n = 0; n < 8; ++n) acc[m][n] = fma(a[m], b[n], acc[m][n]);
  };

  for (int i0 = 0; i0 < d; i0 += CS_BK) {
#pragma unroll
    for (int j = 0; j < CS_BM * CS_BK / 128; ++j) {
      const int e = tid + 128 * j, r = e >> 4, c = e & 15;
      const long long q = q0 + r;
      As[c][r] = q < Q && i0 + c < d ? __ldg(qm + q * d + i0 + c) : 0.0f;
    }
#pragma unroll
    for (int j = 0; j < CS_BN * CS_BK / 128; ++j) {
      const int e = tid + 128 * j, r = e >> 4, c = e & 15;
      const long long n = n0 + r;
      Bs[c][r] = n < N && i0 + c < d ? __ldg(km + n * d + i0 + c) : 0.0f;
    }
    __syncthreads();
    const int kt = min(CS_BK, d - i0);
    if (kt == CS_BK) {
#pragma unroll
      for (int kk = 0; kk < CS_BK; ++kk) step(kk);
    } else {
      for (int kk = 0; kk < kt; ++kk) step(kk);
    }
    __syncthreads();
  }

#pragma unroll
  for (int m = 0; m < 8; ++m) {
    const long long q = q0 + (m < 4 ? ty * 4 + m : 32 + ty * 4 + m - 4);
    if (q >= Q) continue;
    const double qv = qn[q];
    float* row = scores + q * N;
#pragma unroll
    for (int n = 0; n < 8; ++n) {
      const long long c = n0 + (n < 4 ? tx * 4 + n : 64 + tx * 4 + n - 4);
      if (c >= N) continue;
      float s = __double2float_rn(__ddiv_rn(acc[m][n], __dmul_rn(qv, kn[c])));
      if (s != s) s = __int_as_float(0x7fc00000);
      row[c] = s;
    }
  }
}

// The high half of a hit's 64-bit key: order-preserving bits of the score, with -0.0 taken as +0.0 and every NaN as 1,
// below every number (numbers map to 0x007fffff (-inf) and above).  0 is left for a row that is not eligible.
__device__ __forceinline__ unsigned score_key(float s) {
  if (s != s) return 1u;
  unsigned u = __float_as_uint(s);
  if (u == 0x80000000u) u = 0u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// The full key: score_key in the high half, 0xffffffff - index in the low half (the lower index wins a tie), so keys are
// unique and a > b exactly when hit a beats hit b.
__device__ __forceinline__ unsigned long long hit_key(float s, long long idx) {
  return ((unsigned long long)score_key(s) << 32) | (0xffffffffu - (unsigned)idx);
}

// keys[q, w] = score_key(scores[q, w]) when row w beats every neighbour j in [lo_w, hi_w), j != w, else 0.  ranges is an
// optional DEVICE (N, 2) int64 table (null: every row is eligible); each entry is clamped to [0, N].  Neighbours are
// visited outward from w (the range's near end first when w lies outside it) until one beats the row.
__global__ void __launch_bounds__(256)
    search_keys_kernel(const float* __restrict__ scores, long long Q, long long N, const long long* __restrict__ ranges,
                       unsigned* __restrict__ keys) {
  const long long total = Q * N;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
    const long long q = g / N, w = g - q * N;
    const float s = __ldg(scores + g);
    bool eligible = true;
    if (ranges) {
      const long long lo = min(max(__ldg(ranges + 2 * w), 0LL), N);
      const long long hi = min(max(__ldg(ranges + 2 * w + 1), 0LL), N);
      const unsigned long long kw = hit_key(s, w);
      const float* row = scores + q * N;
      // nearest neighbours first: a row that is not a local maximum is usually beaten by an adjacent one, so the scan
      // stops after a step or two even when the neighbourhood spans a whole recording
      long long l = min(w, hi) - 1, r = max(w + 1, lo);
      while (eligible && (l >= lo || r < hi)) {
        if (r < hi && hit_key(__ldg(row + r), r) > kw) eligible = false;
        if (l >= lo && hit_key(__ldg(row + l), l) > kw) eligible = false;
        ++r;
        --l;
      }
    }
    keys[g] = eligible ? score_key(s) : 0u;
  }
}

constexpr int TK_THREADS = 1024;

// Exclusive prefix of a per-thread flag over the block in thread order, and the block's total (all threads call it).
__device__ __forceinline__ unsigned block_prefix(bool flag, unsigned* warp_sums, unsigned* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned ballot = __ballot_sync(0xffffffffu, flag);
  __syncthreads();                                  // warp_sums may still be read by the previous call
  if (lane == 0) warp_sums[warp] = __popc(ballot);
  __syncthreads();
  if (warp == 0) {
    const unsigned v = warp_sums[lane];
    unsigned incl = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const unsigned t = __shfl_up_sync(0xffffffffu, incl, off);
      if (lane >= off) incl += t;
    }
    warp_sums[lane] = incl - v;
    if (lane == 31) *total = incl;
  }
  __syncthreads();
  return warp_sums[warp] + __popc(ballot & ((1u << lane) - 1u));
}

// One block per query row of keys (from search_keys_kernel).  kk = min(k, eligible rows).  A 4-pass radix select (8 bits a
// pass) finds the kk-th largest high key thr and how many rows equal to thr to take, lowest index first; the block then
// walks the row in index order and gathers the kk hits' 64-bit keys into shared memory, bitonic-sorts them descending and
// writes score (read back from scores) and index; slots kk .. k-1 get NaN and -1.
__global__ void __launch_bounds__(TK_THREADS)
    search_topk_kernel(const float* __restrict__ scores, const unsigned* __restrict__ keys, long long N, int k,
                       float* __restrict__ out_score, long long* __restrict__ out_index) {
  __shared__ unsigned hist[256];
  __shared__ unsigned warp_sums[32];
  __shared__ unsigned s_total, s_zeros, s_digit, s_want;
  __shared__ unsigned long long hits[TK_THREADS];
  const int tid = threadIdx.x;
  const long long q = blockIdx.x;
  const unsigned* kr = keys + q * N;
  const float* sr = scores + q * N;

  if (tid == 0) s_zeros = 0;
  __syncthreads();
  unsigned zeros = 0;
  for (long long e = tid; e < N; e += TK_THREADS) zeros += __ldg(kr + e) == 0u;
  atomicAdd(&s_zeros, zeros);
  __syncthreads();
  const long long eligible = N - s_zeros;
  const int kk = (int)min((long long)k, eligible);

  unsigned prefix = 0, mask = 0, want = (unsigned)kk;
  if (kk > 0) {
    for (int shift = 24; shift >= 0; shift -= 8) {
      if (tid < 256) hist[tid] = 0;
      __syncthreads();
      for (long long base = 0; base < N; base += TK_THREADS) {   // whole warps: the tail lanes vote too
        const long long e = base + tid;
        const unsigned key = e < N ? __ldg(kr + e) : 0u;
        const bool in = e < N && (key & mask) == prefix;
        const unsigned active = __ballot_sync(0xffffffffu, in);
        if (in) {
          const unsigned digit = (key >> shift) & 255u;
          const unsigned peers = __match_any_sync(active, digit);
          if ((__ffs(peers) - 1) == (tid & 31)) atomicAdd(&hist[digit], __popc(peers));
        }
      }
      __syncthreads();
      if (tid < 32) {                               // lane l owns bins 8l .. 8l+7; find the bin holding rank `want`
        unsigned c[8], s = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) s += c[j] = hist[tid * 8 + j];
        unsigned suf = s;                           // rows in this lane's bins and every higher one
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const unsigned t = __shfl_down_sync(0xffffffffu, suf, off);
          if (tid + off < 32) suf += t;
        }
        unsigned cum = suf - s;
        if (cum < want && want <= suf) {
          for (int j = 7; j >= 0; --j) {
            if (cum + c[j] >= want) {
              s_digit = tid * 8 + j;
              s_want = want - cum;
              break;
            }
            cum += c[j];
          }
        }
      }
      __syncthreads();
      prefix |= s_digit << shift;
      mask |= 255u << shift;
      want = s_want;
      __syncthreads();
    }
  }
  const unsigned thr = prefix, need = want;        // take every key > thr and the first `need` keys == thr

  unsigned taken = 0, eq_seen = 0;
  for (long long base = 0; base < N && taken < (unsigned)kk; base += TK_THREADS) {
    const long long e = base + tid;
    const unsigned key = e < N ? __ldg(kr + e) : 0u;
    const bool eq = key == thr && e < N;
    const unsigned eq_rank = eq_seen + block_prefix(eq, warp_sums, &s_total);
    eq_seen += s_total;
    const bool take = (key > thr) || (eq && eq_rank < need);
    const unsigned pos = taken + block_prefix(take, warp_sums, &s_total);
    taken += s_total;
    if (take) hits[pos] = ((unsigned long long)key << 32) | (0xffffffffu - (unsigned)e);
  }
  if (tid >= kk) hits[tid] = 0ull;
  for (int size = 2; size <= TK_THREADS; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      const int j = tid ^ stride;
      if (j > tid) {
        const unsigned long long a = hits[tid], b = hits[j];
        if (((tid & size) == 0) ? a < b : a > b) {
          hits[tid] = b;
          hits[j] = a;
        }
      }
    }
  }
  __syncthreads();
  if (tid < k) {
    const long long o = q * k + tid;
    if (tid < kk) {
      const long long idx = 0xffffffffu - (unsigned)(hits[tid] & 0xffffffffull);
      out_index[o] = idx;
      out_score[o] = __ldg(sr + idx);
    } else {
      out_index[o] = -1;
      out_score[o] = __int_as_float(0x7fc00000);
    }
  }
}

}  // namespace
}  // namespace acx

using namespace acx;

extern "C" {

int acx_row_norms(const float* x, long long rows, int d, double* out, void* stream) {
  ACX_CHECK(x && out, ACX_ERR_ARG, "row_norms: null pointer");
  ACX_CHECK(rows >= 1 && rows <= (1LL << 40) && d >= 1, ACX_ERR_ARG, "row_norms: bad sizes rows=%lld d=%d", rows, d);
  row_norms_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(x, rows, d, out);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

int acx_cosine_scores(const float* queries, const double* query_norms, long long Q, const float* keys,
                      const double* key_norms, long long N, int d, float* scores, void* stream) {
  ACX_CHECK(queries && query_norms && keys && key_norms && scores, ACX_ERR_ARG, "cosine_scores: null pointer");
  ACX_CHECK(Q >= 1 && Q <= CS_MAX_Q && N >= 1 && N <= SEARCH_MAX_N && d >= 1, ACX_ERR_ARG,
            "cosine_scores: bad sizes Q=%lld N=%lld d=%d", Q, N, d);
  const dim3 grid((unsigned)((N + CS_BN - 1) / CS_BN), (unsigned)((Q + CS_BM - 1) / CS_BM));
  cosine_scores_kernel<<<grid, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(queries, query_norms, Q, keys, key_norms,
                                                                                 N, d, scores);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

int acx_search_topk_workspace(long long Q, long long N, long long* bytes) {
  ACX_CHECK(bytes, ACX_ERR_ARG, "search_topk_workspace: null pointer");
  ACX_CHECK(Q >= 1 && Q <= SEARCH_MAX_N && N >= 1 && N <= SEARCH_MAX_N, ACX_ERR_ARG,
            "search_topk_workspace: bad sizes Q=%lld N=%lld", Q, N);
  *bytes = Q * N * (long long)sizeof(unsigned);
  return ACX_OK;
}

int acx_search_topk(const float* scores, long long Q, long long N, const long long* ranges, int k, float* out_score,
                    long long* out_index, void* workspace, void* stream) {
  ACX_CHECK(scores && out_score && out_index && workspace, ACX_ERR_ARG, "search_topk: null pointer");
  ACX_CHECK(Q >= 1 && Q <= SEARCH_MAX_N && N >= 1 && N <= SEARCH_MAX_N, ACX_ERR_ARG,
            "search_topk: bad sizes Q=%lld N=%lld", Q, N);
  ACX_CHECK(k >= 1 && k <= SEARCH_MAX_K, ACX_ERR_ARG, "search_topk: k=%d outside [1, %d]", k, SEARCH_MAX_K);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  unsigned* keys = static_cast<unsigned*>(workspace);
  const long long blocks = min((Q * N + 255) / 256, 148LL * 64);
  search_keys_kernel<<<(unsigned)blocks, 256, 0, st>>>(scores, Q, N, ranges, keys);
  ACX_CUDA(cudaGetLastError());
  search_topk_kernel<<<(unsigned)Q, TK_THREADS, 0, st>>>(scores, keys, N, k, out_score, out_index);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

}  // extern "C"
