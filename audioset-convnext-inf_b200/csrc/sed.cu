// Sound event detection: window rows -> activity bins -> timed events (sed.py is the host side and the reference).
#include "common.cuh"

namespace acx {
namespace {

constexpr int SED_C = 527;   // AudioSet classes: one thread per class of a bin (or of a track), class-contiguous

// act[m, c] = (sum over t < n of P[ring_base + (row_first + t) mod ring_cap, c]) / n, the sum taken with plain fp32 adds in
// t order starting from the first row, the division correctly rounded.  tab is a DEVICE (M, 4) int64 table, row m =
// (row_first, n, ring_base, ring_cap).  Every entry is clamped (ring_cap to [1, p_rows], ring_base to [0, p_rows -
// ring_cap], n to [0, ring_cap], row_first reduced mod ring_cap), so no table value reads outside P; a row with n = 0
// gives NaN.  Consecutive threads take consecutive classes of one bin, so every row load is coalesced.
__global__ void __launch_bounds__(256)
    window_activity_kernel(const float* __restrict__ P, long long p_rows, const long long* __restrict__ tab, long long M,
                           float* __restrict__ act) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= M * SED_C) return;
  const long long m = g / SED_C;
  const int c = (int)(g - m * SED_C);
  const long long* e = tab + 4 * m;
  const long long cap = min(max(__ldg(e + 3), 1LL), p_rows);
  const long long base = min(max(__ldg(e + 2), 0LL), p_rows - cap);
  const long long n = min(max(__ldg(e + 1), 0LL), cap);
  long long slot = max(__ldg(e), 0LL);
  if (slot >= cap) slot %= cap;
  float s = __int_as_float(0x7fc00000);
  for (long long t = 0; t < n; ++t) {
    const float v = __ldg(P + (base + slot) * SED_C + c);
    s = t == 0 ? v : __fadd_rn(s, v);
    if (++slot == cap) slot = 0;
  }
  act[g] = n ? __fdiv_rn(s, (float)n) : s;
}

// One (sequence, class) track.  phase: 0 idle, 1 an event is open, 2 an event has ended and may still merge with the next.
// onset / end are the first and last bin of the (merged) event, peak the max of the activity over its bins.
struct Track {
  long long phase, onset, end;
  float peak;
};

template <bool WRITE>
struct Walker {
  Track tr;
  long long R, gap, min_dur, limit, rec;
  int c;
  long long n_out;                 // events emitted so far by this thread
  long long base;                  // WRITE: first output slot of this thread
  long long* out;                  // (4, E): recording, class, onset, offset
  float* out_peak;
  long long E;

  __device__ __forceinline__ long long offset_of(long long end_bin) const { return min((end_bin + 1) * R, limit); }
  __device__ __forceinline__ void emit() {
    const long long on = tr.onset * R, off = offset_of(tr.end);
    if (off - on >= min_dur) {
      if (WRITE) {
        const long long i = base + n_out;
        if (i >= 0 && i < E) {
          out[i] = rec;
          out[E + i] = c;
          out[2 * E + i] = on;
          out[3 * E + i] = off;
          out_peak[i] = tr.peak;
        }
      }
      ++n_out;
    }
    tr.phase = 0;
  }
  // bin j with activity a: the hysteresis state machine of sed.py (reference_events, EventTracks)
  __device__ __forceinline__ void step(long long j, float a, float on_t, float off_t) {
    if (tr.phase == 1) {
      if (a >= off_t) {
        tr.end = j;
        tr.peak = a > tr.peak ? a : tr.peak;
        return;
      }
      tr.phase = 2;                                       // ended at bin j (a NaN ends it too)
    }
    if (tr.phase == 2 && j * R - offset_of(tr.end) >= gap) emit();
    if (a >= on_t) {
      if (tr.phase == 2) {                                // merge: the pending event goes on
        tr.peak = a > tr.peak ? a : tr.peak;
      } else {
        tr.onset = j;
        tr.peak = a;
      }
      tr.phase = 1;
      tr.end = j;
    }
  }
};

// One thread per (sequence, class), g = s * 527 + c.  seq is a DEVICE (S, 6) int64 table, row s = (recording, row0, n_bins,
// j0, limit, close): the sequence's new bins are act rows row0 .. row0 + n_bins - 1, its bins j0 .. j0 + n_bins - 1, bin j
// spans [j R, min((j + 1) R, limit)), and close != 0 ends the sequence (open and pending events are emitted).  State
// (phase, onset, end: (3, S * 527) int64; peak: (S * 527) fp32) carries the track across calls.  WRITE = false counts the
// events each thread emits into slots[g] and changes nothing else; WRITE = true writes them from slot slots[g] (the
// exclusive prefix of the counts) and stores the state.  row0 and n_bins are clamped to act_rows, and an output slot
// outside [0, E) is not written.  The walk is serial in time per track; loads are issued eight bins ahead.
template <bool WRITE>
__global__ void __launch_bounds__(128)
    detect_events_kernel(const float* __restrict__ act, long long act_rows, const long long* __restrict__ seq, int S,
                         const float* __restrict__ on_t, const float* __restrict__ off_t, long long R, long long gap,
                         long long min_dur, long long* __restrict__ state, float* __restrict__ state_peak,
                         long long* __restrict__ slots, long long* __restrict__ out, float* __restrict__ out_peak,
                         long long E) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long n_tracks = (long long)S * SED_C;
  if (g >= n_tracks) return;
  const int s = (int)(g / SED_C);
  const int c = (int)(g - (long long)s * SED_C);
  const long long* e = seq + 6 * (long long)s;
  const long long row0 = min(max(__ldg(e + 1), 0LL), act_rows);
  const long long nb = min(max(__ldg(e + 2), 0LL), act_rows - row0);
  const long long j0 = __ldg(e + 3);
  Walker<WRITE> w;
  w.tr = Track{state[g], state[n_tracks + g], state[2 * n_tracks + g], state_peak[g]};
  w.R = R;
  w.gap = gap;
  w.min_dur = min_dur;
  w.limit = __ldg(e + 4);
  w.rec = __ldg(e);
  w.c = c;
  w.n_out = 0;
  w.base = WRITE ? slots[g] : 0;
  w.out = out;
  w.out_peak = out_peak;
  w.E = E;
  const float on = __ldg(on_t + c), off = __ldg(off_t + c);
  const float* a = act + row0 * SED_C + c;
  for (long long t0 = 0; t0 < nb; t0 += 8) {
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = t0 + u < nb ? __ldg(a + (t0 + u) * SED_C) : 0.0f;
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (t0 + u < nb) w.step(j0 + t0 + u, v[u], on, off);
  }
  if (__ldg(e + 5)) {
    if (w.tr.phase != 0) w.emit();
  } else if (w.tr.phase == 2 && (j0 + nb) * R - w.offset_of(w.tr.end) >= gap) {
    w.emit();                                           // no bin still to come can merge with it
  }
  if (WRITE) {
    state[g] = w.tr.phase;
    state[n_tracks + g] = w.tr.onset;
    state[2 * n_tracks + g] = w.tr.end;
    state_peak[g] = w.tr.peak;
  } else {
    slots[g] = w.n_out;
  }
}

}  // namespace
}  // namespace acx

using namespace acx;

extern "C" {

int acx_window_activity(const float* probs, long long p_rows, const long long* table, long long M, float* act,
                        void* stream) {
  ACX_CHECK(probs && table && act, ACX_ERR_ARG, "window_activity: null pointer");
  ACX_CHECK(p_rows >= 1 && M >= 1 && M <= (1LL << 40) / SED_C, ACX_ERR_ARG, "window_activity: bad sizes p_rows=%lld M=%lld",
            p_rows, M);
  const long long threads = M * SED_C;
  window_activity_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      probs, p_rows, table, M, act);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

int acx_detect_events(const float* act, long long act_rows, const long long* seq, int S, const float* on_threshold,
                      const float* off_threshold, long long resolution, long long merge_gap, long long min_duration,
                      long long* state, float* state_peak, long long* slots, int phase, long long* out, float* out_peak,
                      long long E, void* stream) {
  ACX_CHECK(seq && on_threshold && off_threshold && state && state_peak && slots, ACX_ERR_ARG,
            "detect_events: null pointer");
  ACX_CHECK(act || act_rows == 0, ACX_ERR_ARG, "detect_events: null activity with act_rows=%lld", act_rows);
  ACX_CHECK(phase == 0 || phase == 1, ACX_ERR_ARG, "detect_events: bad phase %d (0 counts, 1 writes)", phase);
  ACX_CHECK(phase == 0 || E == 0 || (out && out_peak), ACX_ERR_ARG, "detect_events: null output");
  ACX_CHECK(S >= 1 && S <= (1 << 30) / SED_C && act_rows >= 0 && act_rows <= (1LL << 40) / SED_C && E >= 0,
            ACX_ERR_ARG, "detect_events: bad sizes S=%d act_rows=%lld E=%lld", S, act_rows, E);
  ACX_CHECK(resolution >= 1 && merge_gap >= 0 && min_duration >= 0, ACX_ERR_ARG,
            "detect_events: bad resolution %lld, merge_gap %lld or min_duration %lld", resolution, merge_gap, min_duration);
  const long long threads = (long long)S * SED_C;
  const unsigned grid = (unsigned)((threads + 127) / 128);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (phase == 0)
    detect_events_kernel<false><<<grid, 128, 0, st>>>(act, act_rows, seq, S, on_threshold, off_threshold, resolution,
                                                      merge_gap, min_duration, state, state_peak, slots, out, out_peak, E);
  else
    detect_events_kernel<true><<<grid, 128, 0, st>>>(act, act_rows, seq, S, on_threshold, off_threshold, resolution,
                                                     merge_gap, min_duration, state, state_peak, slots, out, out_peak, E);
  ACX_CUDA(cudaGetLastError());
  return ACX_OK;
}

}  // extern "C"
