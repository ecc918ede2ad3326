// Shared host/device helpers for libacx (B200 / sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <atomic>

#include "../../include/acx.h"

namespace acx {

// ---- error plumbing (thread-local last error; no exceptions cross the C ABI) -------------
void set_error(const char* fmt, ...);
const char* last_error();

#define ACX_CHECK(cond, code, ...)                  \
  do {                                              \
    if (!(cond)) {                                  \
      ::acx::set_error(__VA_ARGS__);                \
      return (code);                                \
    }                                               \
  } while (0)

#define ACX_CUDA(expr)                                                              \
  do {                                                                              \
    cudaError_t _e = (expr);                                                        \
    if (_e != cudaSuccess) {                                                        \
      ::acx::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),      \
                       __FILE__, __LINE__);                                         \
      return ACX_ERR_CUDA;                                                          \
    }                                                                               \
  } while (0)

// Opt a kernel into more than 48 KB of dynamic shared memory.  The attribute is PER DEVICE, so it is remembered with one
// bit per device (a process that drives several GPUs would otherwise configure only the first one it used).
#define ACX_SET_MAX_SMEM(kern, bytes)                                                               \
  do {                                                                                              \
    static std::atomic<unsigned long long> acx_done_{0};   /* host threads may drive different GPUs at once */    \
    int acx_dev_ = 0;                                                                               \
    ACX_CUDA(cudaGetDevice(&acx_dev_));                                                             \
    if (acx_dev_ >= 64 || !((acx_done_.load(std::memory_order_acquire) >> acx_dev_) & 1ull)) {      \
      ACX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (bytes)));   \
      if (acx_dev_ < 64) acx_done_.fetch_or(1ull << acx_dev_, std::memory_order_release);           \
    }                                                                                               \
  } while (0)

// SM count of the current device (cached per device; the persistent grids are sized from it, never hard-coded)
static inline int sm_count() {
  static std::atomic<int> cached[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev < 64) {
    const int c = cached[dev].load(std::memory_order_relaxed);
    if (c > 0) return c;
  }
  int sms = 0;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) return 148;
  if (dev < 64) cached[dev].store(sms, std::memory_order_relaxed);
  return sms;
}

#ifndef ACX_PDL_DEFAULT
#define ACX_PDL_DEFAULT 7   /* GEMM + fused MLP + tensor-core conv: measured -2 % step time; with the small kernels included the gain is lost (tools/ab_pdl.py) */
#endif
// ---- programmatic dependent launch ----------------------------------------------------------------------------------
// The ~68 kernels of a forward run back to back on one stream.  Launched with the programmatic-stream-serialization
// attribute, kernel i+1's CTAs are scheduled as soon as every CTA of kernel i has executed pdl_trigger() and an SM has
// room: their prologue (barrier init, TMEM allocation, weight preload, band build -- nothing that depends on kernel i)
// runs under kernel i's tail, and they block in pdl_wait() until kernel i has completed and its writes are visible.
// Rules every kernel on the path follows:
//   * pdl_trigger() comes AFTER the CTA has acquired everything it will ever need (TMEM): a dependent CTA that became
//     co-resident earlier could take the TMEM columns this CTA still has to allocate and then wait for it forever;
//   * pdl_wait() comes before the first access (read OR write) to any buffer another kernel of the stream touches;
//     only weights / constants may be read above it.
// Without the attribute (ACX_PDL=0, or a launch that follows a non-kernel stream operation) both are no-ops.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// which launches carry the attribute: ACX_PDL is a bit mask over the kernel families (A/B experiments); 0 = none
enum PdlKind { PDL_GEMM = 1, PDL_MLP = 2, PDL_DWTC = 4, PDL_STATS = 8, PDL_SMALL = 16 };
static inline bool pdl_enabled(int kind) {      // read per launch: a captured graph keeps what was set at capture time
  const char* e = getenv("ACX_PDL");
  return ((e ? atoi(e) : ACX_PDL_DEFAULT) & kind) != 0;
}

// cudaLaunchKernelEx with the programmatic-stream-serialization attribute (and optionally a cluster dimension)
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, int cluster_x,
                                     int kind, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  unsigned na = 0;
  if (cluster_x > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = cluster_x;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl_enabled(kind)) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- device helpers ---------------------------------------------------------------------
using bf16 = __nv_bfloat16;

template <typename T> struct Pair;          // two consecutive channels
template <> struct Pair<float> {
  using type = float2;
  __device__ static __forceinline__ float2 unpack(float2 v) { return v; }
  __device__ static __forceinline__ float2 pack(float a, float b) { return make_float2(a, b); }
};
template <> struct Pair<bf16> {
  using type = uint32_t;
  // bf16 -> fp32 is a 16-bit shift: two ALU ops per pair, no conversion pipe.
  __device__ static __forceinline__ float2 unpack(uint32_t v) {
    return make_float2(__uint_as_float(v << 16), __uint_as_float(v & 0xffff0000u));
  }
  __device__ static __forceinline__ uint32_t pack(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
};

__device__ __forceinline__ float to_float(float v) { return v; }
__device__ __forceinline__ float to_float(bf16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_float(float v);
template <> __device__ __forceinline__ float from_float<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_float<bf16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Exact (erf) GELU -- nn.GELU() default, reference convnext.py:65.
__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}

// ---- tensor-core-path GELU on a register tile -----------------------------------------------------------------
// 0.5 x (1 + tanh(x (a + b x^2 + c x^4))) with MUFU.TANH; (a, b, c) are a minimax re-fit against the EXACT erf GELU the
// reference uses (nn.GELU(), convnext.py:65): max |err| 2.6e-5 over all x (textbook tanh-GELU: 4.7e-4), ~10x below the
// bf16 rounding applied to the result; x^2 is clamped at 50 (tanh saturated) so the negative x^4 term cannot flip the
// sign for |x| > 11.  Checked on the CPU by tests/test_host_logic.py::test_gelu_fit_against_exact_erf.
// All arithmetic is packed fp32x2 (FADD2 / FMUL2 / FFMA2 of sm_100).  The "twice" form returns 2 * gelu
// (= x + x tanh(.)): the fused MLP folds the missing 0.5 into its layer-scale vector (exact: powers of two).
//
// The GELU is split into three stages for a column pair -- A: bias + polynomial (FMA pipe), T: 2 x MUFU.TANH (XU
// pipe), C: x + x t (FMA pipe) -- so that callers can software-pipeline T of one group of columns against A of the
// next.  History (clock traces + ncu, profiles/): written pair by pair the compiler serialised each pair's 8-deep chain
// (~0.15 IPC per epilogue warp); written stage by stage over a whole tile, the two epilogue warps that share a
// scheduler sat in the same stage at the same time and the XU and FMA pipes alternated instead of overlapping
// (~2.0 k cycles per 128 x 128 chunk against a 1.0 k XU floor).
struct GeluPair {
  unsigned long long x, u;   // packed fp32x2
};
// Every stage instruction is `asm volatile` in a hand-chosen order: left to itself the compiler re-clusters them into
// long FMA-only and MUFU-only runs (seen in SASS), which is what the software pipeline is there to avoid.  Because a
// warp issues in order, the order below keeps dependent instructions >= 4 issue slots apart (four column pairs advance
// in lock step through the 6-deep polynomial chain) and sprinkles the other group's MUFUs in between.
__device__ __forceinline__ unsigned long long f2_pack(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void gelu_op_tanh(GeluPair& g) {
  asm volatile(
      "{\n\t.reg .f32 lo, hi;\n\tmov.b64 {lo, hi}, %0;\n\ttanh.approx.f32 lo, lo;\n\ttanh.approx.f32 hi, hi;\n\t"
      "mov.b64 %0, {lo, hi};\n\t}"
      : "+l"(g.u));
}
// stage T on t[0..4) (if kT) interleaved with stage A on a[0..4) (if kA): acc = 8 fp32 accumulator words, sbias_addr =
// shared-space address of their 8 biases.  (Fetching the biases a whole step ahead into 8 more registers was tried:
// the kernel sits at the 128-register cap and got 5 % slower.)
// kFold: the accumulator is G = v . (W1 diag(ln_w))^T of the UN-normalised conv output v, and the LayerNorm (CX:78) is
// applied here as a rank-1 correction:  pre = rstd_p * G + (nmr_p * s_j + b1'_j)   with  nmr_p = -mean_p * rstd_p,
// s_j = sum_c W1'[j, c],  b1' = b1 + W1 ln_b   (fold = {rstd, rstd}, {nmr, nmr} packed; s sits `s_off` bytes behind
// the biases in shared memory).  One extra packed FMA per column pair instead of a LayerNorm pass over the tensor.
struct LnFold {
  unsigned long long rstd2, nmr2;
  uint32_t sb1_base, sbs_base;   // smem addresses of b1[] and of the interleaved {b1[2q], b1[2q+1], s[2q], s[2q+1]} array:
};                               // ONE 16-byte load brings a column pair's biases and s (a second 8-byte load cost 9 %)
template <bool kT, bool kA, bool kFold = false>
__device__ __forceinline__ void gelu_stage_ta4(GeluPair* t, GeluPair* a, const uint32_t* acc, uint32_t sbias_addr,
                                               const LnFold fold = LnFold{}) {
  const unsigned long long k50 = f2_pack(50.0f, 50.0f);
  const unsigned long long kc = f2_pack(-3.51516788e-04f, -3.51516788e-04f);
  const unsigned long long kb = f2_pack(3.70056460e-02f, 3.70056460e-02f);
  const unsigned long long ka = f2_pack(7.97507884e-01f, 7.97507884e-01f);
  unsigned long long q[4], p[4];
  if (kT) gelu_op_tanh(t[0]);
  if (kA) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float2 b;
      if (kFold) {
        float2 sj;
        asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
            : "=f"(b.x), "=f"(b.y), "=f"(sj.x), "=f"(sj.y)
            : "r"(fold.sbs_base + 2 * (sbias_addr - fold.sb1_base) + 16 * i));
        unsigned long long tt;
        asm volatile("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(tt) : "l"(fold.nmr2), "l"(f2_pack(sj.x, sj.y)), "l"(f2_pack(b.x, b.y)));
        asm volatile("fma.rn.f32x2 %0, %1, %2, %3;"
                     : "=l"(a[i].x)
                     : "l"(fold.rstd2), "l"(f2_pack(__uint_as_float(acc[2 * i]), __uint_as_float(acc[2 * i + 1]))), "l"(tt));
      } else {
        asm("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(b.x), "=f"(b.y) : "r"(sbias_addr + 8 * i));
        asm volatile("add.rn.f32x2 %0, %1, %2;"
                     : "=l"(a[i].x)
                     : "l"(f2_pack(__uint_as_float(acc[2 * i]), __uint_as_float(acc[2 * i + 1]))), "l"(f2_pack(b.x, b.y)));
      }
    }
  }
  if (kT) gelu_op_tanh(t[1]);
  if (kA) {
#pragma unroll
    for (int i = 0; i < 4; ++i) asm volatile("mul.rn.f32x2 %0, %1, %1;" : "=l"(q[i]) : "l"(a[i].x));
#pragma unroll
    for (int i = 0; i < 4; ++i)
      asm volatile(
          "{\n\t.reg .f32 lo, hi, c;\n\tmov.b64 {lo, hi}, %0;\n\tmov.b64 {c, _}, %1;\n\t"
          "min.f32 lo, lo, c;\n\tmin.f32 hi, hi, c;\n\tmov.b64 %0, {lo, hi};\n\t}"
          : "+l"(q[i])
          : "l"(k50));
  }
  if (kT) gelu_op_tanh(t[2]);
  if (kA) {
#pragma unroll
    for (int i = 0; i < 4; ++i) asm volatile("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(p[i]) : "l"(q[i]), "l"(kc), "l"(kb));
  }
  if (kT) gelu_op_tanh(t[3]);
  if (kA) {
#pragma unroll
    for (int i = 0; i < 4; ++i) asm volatile("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(q[i]) : "l"(q[i]), "l"(p[i]), "l"(ka));
#pragma unroll
    for (int i = 0; i < 4; ++i) asm volatile("mul.rn.f32x2 %0, %1, %2;" : "=l"(a[i].u) : "l"(a[i].x), "l"(q[i]));
  }
}
// stage C on 8 pairs: 2 * gelu (= x + x tanh(.)) packed to bf16x2; the 8 FMAs first, then the 8 conversions
__device__ __forceinline__ void gelu_stage_c8_twice_bf16(const GeluPair* g, uint32_t* pk) {
  unsigned long long o[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) asm volatile("fma.rn.f32x2 %0, %1, %2, %1;" : "=l"(o[i]) : "l"(g[i].x), "l"(g[i].u));
#pragma unroll
  for (int i = 0; i < 8; ++i)
    asm volatile("{\n\t.reg .f32 lo, hi;\n\tmov.b64 {lo, hi}, %1;\n\tcvt.rn.bf16x2.f32 %0, hi, lo;\n\t}"
                 : "=r"(pk[i])
                 : "l"(o[i]));
}

// Drop-in for bias_gelu_tile<16, kTwice> built from the stages above: T of pairs [4k, 4k+4) is interleaved with A of
// pairs [4k+4, 4k+8), so each warp's instruction stream mixes XU and FMA work instead of alternating long phases.
template <bool kTwice, bool kFold = false>
__device__ __forceinline__ void bias_gelu_tile16_sp(const uint32_t* __restrict__ acc /*[32] fp32 bits*/,
                                                    const float* __restrict__ sbias /*smem*/, float2 (&out)[16],
                                                    const LnFold fold = LnFold{}) {
  GeluPair g[16];
  const uint32_t sb = static_cast<uint32_t>(__cvta_generic_to_shared(sbias));
  gelu_stage_ta4<false, true, kFold>(nullptr, g, acc, sb, fold);
  gelu_stage_ta4<true, true, kFold>(g, g + 4, acc + 8, sb + 32, fold);
  gelu_stage_ta4<true, true, kFold>(g + 4, g + 8, acc + 16, sb + 64, fold);
  gelu_stage_ta4<true, true, kFold>(g + 8, g + 12, acc + 24, sb + 96, fold);
  gelu_stage_ta4<true, false>(g + 12, nullptr, nullptr, 0);
  const unsigned long long khalf = f2_pack(0.5f, 0.5f);
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    unsigned long long o, x = g[i].x;
    if (!kTwice) asm volatile("mul.rn.f32x2 %0, %1, %2;" : "=l"(x) : "l"(g[i].x), "l"(khalf));
    asm volatile("fma.rn.f32x2 %0, %1, %2, %1;" : "=l"(o) : "l"(x), "l"(g[i].u));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(out[i].x), "=f"(out[i].y) : "l"(o));
  }
}

}  // namespace acx
