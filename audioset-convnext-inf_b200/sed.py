"""Sound event detection: from window tags to "what happened when" (dog bark from 03:12:05 to 03:12:09 on mic 17).

sed.detect(model.forward_windows(...), Detection(...)) turns the overlapping window rows of long recordings into an
activity track per class on a time grid and into timed events; ConvNeXt.open_stream(..., detection=...) does the same as
live audio arrives, bit for bit.  Times are in 32 kHz samples of the (resampled) recording, as the windows' "start" is.

Semantics (the numpy reference below is these definitions written out literally):

  Input: the dict forward_windows returns, or a stream's rows.  Only "clipwise_output", "recording", "start" and
  "length" are read.  Rows are recording-major with start ascending.  The length n_r of recording r is max(start +
  length) over its rows (a plan_windows plan always ends at the recording's last sample).

  Activity: resolution R cuts recording r into bins j = 0 .. ceil(n_r / R) - 1; bin j spans [j R, min((j + 1) R, n_r)).
  W_j are the recording's windows that intersect the bin (start < bin_end and start + length > bin_start), in row
  order, and
      a[j, c] = __fdiv_rn(s, |W_j|),  s = the float32 sum of clipwise_output[w, c] over W_j, plain adds in row order
  starting from the first row.  R >= n_r gives one bin: the recording-level tags (the mean of all its windows).  A bin
  no window intersects (possible only when hop > window) raises ValueError.

  Events, per (recording, class) track, with thresholds on[c] >= off[c]: a raw event opens at a bin with a >= on when
  none is open, stays open while a >= off and ends at the first bin where !(a >= off) (a NaN ends it); its onset is its
  first bin's start and its offset the end of its last bin.  Consecutive events of a class merge when next.onset -
  prev.offset < merge_gap_samples; after merging an event is kept when offset - onset >= min_duration_samples.  peak is
  the max of a over the event's bins (bins in a merge gap are below off, so the max over the whole span is the same).
  Events are ordered (recording, class, onset).

Device work: acx_window_activity computes the bins from a host-built (M, 4) table of row ranges (the W_j), and
acx_detect_events walks every track's bins in one thread, in a count phase and a write phase.  Reading the event count
back to size the outputs costs one device-to-host synchronisation per call."""
import numbers

import numpy as np
import torch

from . import _native
from .engine import N_CLASSES
from .windows import check_rows

ACTIVITY_KEYS = ("activity", "recording", "start", "length")
EVENT_KEYS = ("recording", "class", "onset", "offset", "peak")


def _count(v, name, low):
    if isinstance(v, bool) or not isinstance(v, numbers.Integral) or int(v) < low:
        raise ValueError(f"{name} = {v!r}: expected an int >= {low}")
    return int(v)


def _thresholds(v, name):
    a = v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
    if a.dtype == bool or not (np.issubdtype(a.dtype, np.floating) or np.issubdtype(a.dtype, np.integer)):
        raise ValueError(f"{name} must be a number or {N_CLASSES} numbers, got dtype {a.dtype}")
    if a.shape not in ((), (N_CLASSES,)):
        raise ValueError(f"{name} must be a scalar or have shape ({N_CLASSES},), got {a.shape}")
    a = np.broadcast_to(a.astype(np.float32), (N_CLASSES,)).copy()
    if not np.isfinite(a).all():
        raise ValueError(f"{name} must be finite")
    return a


class Detection:
    """What to detect: bins of resolution_samples (32 kHz samples, >= 1), thresholds onset_threshold >=
    offset_threshold (each a float32 scalar or one per class, finite; offset_threshold=None means the onset threshold),
    and the merge gap and minimum duration in samples (ints >= 0).  Checked when built; raises ValueError."""

    def __init__(self, resolution_samples, onset_threshold, offset_threshold=None, min_duration_samples=0,
                 merge_gap_samples=0):
        self.resolution = _count(resolution_samples, "resolution_samples", 1)
        self.on = _thresholds(onset_threshold, "onset_threshold")
        self.off = self.on.copy() if offset_threshold is None else _thresholds(offset_threshold, "offset_threshold")
        bad = np.flatnonzero(self.off > self.on)
        if bad.size:
            raise ValueError(f"offset_threshold exceeds onset_threshold for class {int(bad[0])}")
        self.min_duration = _count(min_duration_samples, "min_duration_samples", 0)
        self.merge_gap = _count(merge_gap_samples, "merge_gap_samples", 0)
        self._dev = {}

    def device_thresholds(self, device):
        key = str(device)
        if key not in self._dev:
            self._dev[key] = torch.from_numpy(np.stack([self.on, self.off])).to(device)
        return self._dev[key]


# ---- host planning ------------------------------------------------------------------------------------------------------
def bin_ranges(starts, ends, j0, j1, R, n):
    """Rows of W_j for bins j0 .. j1 - 1 of a recording of n samples whose windows, in row order, have the given starts
    (ascending) and ends (non-decreasing): (first, count) arrays, the rows [first, first + count).  A window intersects
    bin j when start < bin_end and end > bin_start, so W_j is a contiguous run of rows."""
    j = np.arange(j0, j1, dtype=np.int64)
    first = np.searchsorted(ends, j * R, side="right")
    last = np.searchsorted(starts, np.minimum((j + 1) * R, n), side="left")
    return first.astype(np.int64), (last - first).astype(np.int64)


def _host_rows(windows):
    """The windows dict checked on the host: (probs on the device, recording, start, length as numpy int64).
    ValueError for missing keys, mismatched row counts, or rows out of recording-major / start-ascending order."""
    if not isinstance(windows, dict):
        raise ValueError("detect takes the dict forward_windows returns")
    missing = [k for k in ("clipwise_output", "recording", "start", "length") if k not in windows]
    if missing:
        raise ValueError(f"windows dict lacks {missing}")
    probs = windows["clipwise_output"]
    if not isinstance(probs, torch.Tensor) or probs.dim() != 2 or probs.shape[1] != N_CLASSES \
            or probs.dtype != torch.float32:
        raise ValueError(f"clipwise_output must be a (N, {N_CLASSES}) float32 tensor")
    rec, start, length = check_rows(windows, probs.shape[0], "clipwise_output")
    return probs.contiguous(), rec, start, length


def plan_bins(rec, start, length, R):
    """Every bin of every recording, checked before any launch.  Returns (table (M, 4) int64 for acx_window_activity
    on the rows themselves, bins {recording, start, length} (M,) int64, seq (S, 6) int64 for acx_detect_events over the
    recordings present, fresh state and closed).  ValueError for a bin no window intersects."""
    N = len(rec)
    edges = np.flatnonzero(np.diff(rec)) + 1
    lo = np.concatenate([[0], edges]).astype(np.int64)
    hi = np.concatenate([edges, [N]]).astype(np.int64)
    tables, b_rec, b_start, b_len, seq = [], [], [], [], []
    row0 = 0
    for a, b in zip(lo.tolist(), hi.tolist()):
        n = int((start[a:b] + length[a:b]).max())
        nb = -(-n // R)
        first, count = bin_ranges(start[a:b], start[a:b] + length[a:b], 0, nb, R, n)
        if (count < 1).any():
            j = int(np.flatnonzero(count < 1)[0])
            raise ValueError(f"bin {j} of recording {int(rec[a])} ([{j * R}, {min((j + 1) * R, n)})) is covered by no "
                             "window: the hop exceeds the window")
        tables.append(np.stack([first + a, count, np.zeros_like(count), np.full_like(count, N)], axis=1))
        j = np.arange(nb, dtype=np.int64)
        b_rec.append(np.full(nb, rec[a], dtype=np.int64))
        b_start.append(j * R)
        b_len.append(np.minimum((j + 1) * R, n) - j * R)
        seq.append((int(rec[a]), row0, nb, 0, n, 1))
        row0 += nb
    bins = {"recording": np.concatenate(b_rec), "start": np.concatenate(b_start), "length": np.concatenate(b_len)}
    return np.concatenate(tables).astype(np.int64), bins, np.array(seq, dtype=np.int64).reshape(-1, 6)


# ---- device work --------------------------------------------------------------------------------------------------------
def window_activity(probs, table):
    """acx_window_activity: (M, 527) float32 bins from rows of probs ((P, 527) float32 on the device) given by the (M, 4)
    int64 host table."""
    dev = probs.device
    M = len(table)
    act = torch.empty(M, N_CLASSES, dtype=torch.float32, device=dev)
    if M:
        tab = torch.from_numpy(np.ascontiguousarray(table)).pin_memory().to(dev, non_blocking=True)
        st = torch.cuda.current_stream(dev).cuda_stream
        _native.call("acx_window_activity", probs.data_ptr(), probs.shape[0], tab.data_ptr(), M, act.data_ptr(), st)
    return act


def new_state(n_seq, device):
    """Fresh event state of n_seq sequences: (3, n_seq * 527) int64 phase / onset bin / last bin and (n_seq * 527) float32
    peak, all zero (idle)."""
    return (torch.zeros(3, n_seq * N_CLASSES, dtype=torch.int64, device=device),
            torch.zeros(n_seq * N_CLASSES, dtype=torch.float32, device=device))


def detect_events(act, seq, detection, state):
    """acx_detect_events over the sequences of the (S, 6) int64 host table seq (rows (recording, row0, n_bins, j0, limit,
    close) into act), carrying `state` (new_state(S)).  Count phase, exclusive scan, one device-to-host read of the
    total, write phase.  Returns the events dict, ordered (sequence, class, onset)."""
    dev = state[0].device
    S = len(seq)
    st = torch.cuda.current_stream(dev).cuda_stream
    thr = detection.device_thresholds(dev)
    seq_d = torch.from_numpy(np.ascontiguousarray(seq)).pin_memory().to(dev, non_blocking=True)
    slots = torch.empty(S * N_CLASSES, dtype=torch.int64, device=dev)
    args = (act.data_ptr() if act.numel() else 0, act.shape[0], seq_d.data_ptr(), S, thr[0].data_ptr(), thr[1].data_ptr(),
            detection.resolution, detection.merge_gap, detection.min_duration, state[0].data_ptr(), state[1].data_ptr(),
            slots.data_ptr())
    _native.call("acx_detect_events", *args, 0, 0, 0, 0, st)
    counts = slots.clone()
    torch.cumsum(counts, 0, out=slots)
    E = int(slots[-1])                                           # the one device-to-host synchronisation
    slots.sub_(counts)
    out = torch.empty(4, E, dtype=torch.int64, device=dev)
    peak = torch.empty(E, dtype=torch.float32, device=dev)
    _native.call("acx_detect_events", *args, 1, out.data_ptr() if E else 0, peak.data_ptr() if E else 0, E, st)
    return {"recording": out[0], "class": out[1], "onset": out[2], "offset": out[3], "peak": peak}


def detect(windows, detection):
    """Activity tracks and timed events of the recordings in `windows` (the dict forward_windows returns):
    {"activity": {"activity" (M, 527) float32, "recording", "start", "length" (M,) int64 per bin, recording-major with
    start ascending}, "events": {"recording", "class", "onset", "offset" (E,) int64, "peak" (E,) float32, ordered
    (recording, class, onset)}}, on the windows' device; see the module docstring for the definitions.  The dict is
    checked on the host before any launch (keys, row counts, row order, every bin covered); a failure raises ValueError
    and launches nothing.  One device-to-host synchronisation (the event count)."""
    if not isinstance(detection, Detection):
        raise ValueError("detection must be a sed.Detection")
    probs, rec, start, length = _host_rows(windows)
    dev = probs.device
    if not len(rec):
        if not probs.is_cuda:
            raise ValueError("clipwise_output must be on a CUDA device: detection runs on the GPU")
        empty = torch.zeros(0, dtype=torch.int64, device=dev)
        return {"activity": {"activity": torch.empty(0, N_CLASSES, dtype=torch.float32, device=dev),
                             "recording": empty, "start": empty, "length": empty},
                "events": {"recording": empty, "class": empty, "onset": empty, "offset": empty,
                           "peak": torch.empty(0, dtype=torch.float32, device=dev)}}
    table, bins, seq = plan_bins(rec, start, length, detection.resolution)
    if not probs.is_cuda:
        raise ValueError("clipwise_output must be on a CUDA device: detection runs on the GPU")
    act = window_activity(probs, table)
    events = detect_events(act, seq, detection, new_state(len(seq), dev))
    activity = {"activity": act}
    activity.update({k: torch.from_numpy(v).to(dev) for k, v in bins.items()})
    return {"activity": activity, "events": events}


# ---- numpy reference ----------------------------------------------------------------------------------------------------
def reference_activity(probs, rec, start, length, R):
    """The activity definition written out: for every bin, every row of its recording tested for intersection, the
    intersecting rows' float32 values added in row order from the first, then one float32 division."""
    probs = np.asarray(probs, dtype=np.float32)
    rows, b_rec, b_start, b_len = [], [], [], []
    for r in sorted(set(rec.tolist())):
        idx = [i for i in range(len(rec)) if rec[i] == r]
        n = max(int(start[i] + length[i]) for i in idx)
        for j in range(-(-n // R)):
            bs, be = j * R, min((j + 1) * R, n)
            s, count = None, 0
            for i in idx:
                if start[i] < be and start[i] + length[i] > bs:
                    s = probs[i].copy() if s is None else (s + probs[i]).astype(np.float32)
                    count += 1
            if count == 0:
                raise ValueError(f"bin {j} of recording {r} is covered by no window")
            rows.append((s / np.float32(count)).astype(np.float32))
            b_rec.append(r)
            b_start.append(bs)
            b_len.append(be - bs)
    i64 = lambda v: np.array(v, dtype=np.int64)                  # noqa: E731
    return {"activity": np.array(rows, dtype=np.float32).reshape(-1, N_CLASSES), "recording": i64(b_rec),
            "start": i64(b_start), "length": i64(b_len)}


def reference_events(activity, detection):
    """The event definitions written out on a reference_activity result: raw events per track, then merging, then the
    duration filter.  Returns numpy arrays keyed like detect's events, ordered (recording, class, onset)."""
    a, rec, start, length = (activity[k] for k in ("activity", "recording", "start", "length"))
    out = {k: [] for k in EVENT_KEYS}
    for r in sorted(set(rec.tolist())):
        idx = np.flatnonzero(rec == r)
        for c in range(N_CLASSES):
            on, off = detection.on[c], detection.off[c]
            raw, cur = [], None                                  # cur: [onset, offset, peak]
            for i in idx:
                v = a[i, c]
                if cur is not None:
                    if v >= off:
                        cur[1] = start[i] + length[i]
                        cur[2] = max(cur[2], v)
                        continue
                    raw.append(cur)
                    cur = None
                if v >= on:
                    cur = [start[i], start[i] + length[i], v]
            if cur is not None:
                raw.append(cur)
            merged = []
            for e in raw:
                if merged and e[0] - merged[-1][1] < detection.merge_gap:
                    merged[-1] = [merged[-1][0], e[1], max(merged[-1][2], e[2])]
                else:
                    merged.append(list(e))
            for onset, offset, peak in merged:
                if offset - onset >= detection.min_duration:
                    for k, v in zip(EVENT_KEYS, (r, c, onset, offset, peak)):
                        out[k].append(v)
    return {k: np.array(v, dtype=np.float32 if k == "peak" else np.int64) for k, v in out.items()}


class EventTracks:
    """The state machine of acx_detect_events in numpy, carried across calls: step(a (nb, 527), j0, limit, close) walks
    new bins j0 .. j0 + nb - 1 of one sequence and returns the events that became final, as (class, onset, offset,
    peak) tuples ordered (class, onset).  Fed a recording's bins in any split and then closed, it gives
    reference_events of that recording."""

    def __init__(self, detection):
        self.d = detection
        self.phase = np.zeros(N_CLASSES, dtype=np.int64)
        self.onset = np.zeros(N_CLASSES, dtype=np.int64)
        self.end = np.zeros(N_CLASSES, dtype=np.int64)
        self.peak = np.zeros(N_CLASSES, dtype=np.float32)

    def step(self, a, j0, limit, close):
        R, gap = self.d.resolution, self.d.merge_gap
        out = []
        for c in range(N_CLASSES):
            ph, on_b, eb, pk = int(self.phase[c]), int(self.onset[c]), int(self.end[c]), self.peak[c]
            on, off = self.d.on[c], self.d.off[c]

            def emit():
                onset, offset = on_b * R, min((eb + 1) * R, limit)
                if offset - onset >= self.d.min_duration:
                    out.append((c, onset, offset, pk))

            for t in range(len(a)):
                j, v = j0 + t, a[t, c]
                if ph == 1:
                    if v >= off:
                        eb, pk = j, max(pk, v)
                        continue
                    ph = 2
                if ph == 2 and j * R - min((eb + 1) * R, limit) >= gap:
                    emit()
                    ph = 0
                if v >= on:
                    if ph == 2:
                        pk = max(pk, v)
                    else:
                        on_b, pk = j, v
                    ph, eb = 1, j
            if close:
                if ph:
                    emit()
                ph = 0
            elif ph == 2 and (j0 + len(a)) * R - min((eb + 1) * R, limit) >= gap:
                emit()
                ph = 0
            self.phase[c], self.onset[c], self.end[c], self.peak[c] = ph, on_b, eb, pk
        return out
