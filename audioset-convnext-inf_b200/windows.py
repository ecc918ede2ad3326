"""Sliding-window tagging of long recordings (a podcast, a day of soundscape monitoring, a film soundtrack).

An AudioSet tagger is applied to a long recording the way it was trained: on windows of `window` samples (10 s) at a hop,
each window tagged as a clip of its own.  The windows are never copied out of the recording: ConvNeXt.forward_windows lays
the recordings end to end in one device buffer, and the prep kernels (acx_wave_prep_windows, acx_frame_fold_windows) read
window b at its 64-bit offset into that buffer.  Everything after the prep is the ordinary batch path.

The plan is pure host logic and is checked in full before anything is launched."""
import collections

import numpy as np
import torch

from .engine import MIN_RAGGED_LEN
from .extract import ragged_batches

# recording, start, length, offset: (N,) int64 CPU tensors in plan order (recording-major, start ascending).  offset is the
# window's first sample in the recordings laid end to end in input order (the buffer forward_windows builds).
WindowPlan = collections.namedtuple("WindowPlan", "recording start length offset window")


def plan_windows(lengths, window=320000, hop=32000):
    """Windows of `window` samples at `hop` over recordings of the given lengths (samples).

    A recording shorter than the window gets one window (0, n) at its own length (run as a ragged clip); one of exactly
    `window` samples is one ordinary window.  Longer ones get windows at 0, hop, 2 hop, ... while start + window <= n, and,
    if the last of those ends before n, one end-aligned window (n - window, window): every sample is covered by a
    full-length window and the model is never shown zero padding.  hop > window leaves gaps, which are never read.
    Raises ValueError for window < MIN_RAGGED_LEN, hop < 1 or a recording shorter than MIN_RAGGED_LEN."""
    window, hop = int(window), int(hop)
    if window < MIN_RAGGED_LEN:
        raise ValueError(f"window_samples={window} is shorter than the shortest clip the model takes ({MIN_RAGGED_LEN} samples)")
    if hop < 1:
        raise ValueError(f"hop_samples must be at least 1, got {hop}")
    lengths = [int(n) for n in lengths]
    for r, n in enumerate(lengths):
        if n < MIN_RAGGED_LEN:
            raise ValueError(f"recording {r} has {n} samples; the shortest the model takes is {MIN_RAGGED_LEN}")
    recs, starts, lens, offs = [], [], [], []
    base = 0
    for r, n in enumerate(lengths):
        if n <= window:
            s = np.zeros(1, dtype=np.int64)
            ln = n
        else:
            s = np.arange(0, n - window + 1, hop, dtype=np.int64)
            if s[-1] + window < n:
                s = np.append(s, np.int64(n - window))
            ln = window
        recs.append(np.full(s.size, r, dtype=np.int64))
        starts.append(s)
        lens.append(np.full(s.size, ln, dtype=np.int64))
        offs.append(s + base)
        base += n

    def cat(parts):
        return torch.from_numpy(np.concatenate(parts)) if parts else torch.zeros(0, dtype=torch.int64)

    return WindowPlan(cat(recs), cat(starts), cat(lens), cat(offs), window)


def window_batches(plan, chunk):
    """[(canvas, lengths or None, indices)] in execution order.  Full-length windows go `chunk` at a time on a canvas of
    plan.window with lengths None: they run NON-ragged, so they replay the CUDA graph forward_all captures for
    (chunk, window).  Own-length windows (recordings shorter than the window) are grouped by extract.ragged_batches and run
    ragged with their lengths.  indices are rows of the plan; results are scattered back to them."""
    length = plan.length.tolist()
    full = [i for i, n in enumerate(length) if n == plan.window]
    short = [i for i, n in enumerate(length) if n != plan.window]
    out = [(plan.window, None, full[b0:b0 + chunk]) for b0 in range(0, len(full), chunk)]
    for canvas, idx in ragged_batches([length[i] for i in short], chunk):
        rows = [short[j] for j in idx]
        out.append((canvas, [length[i] for i in rows], rows))
    return out


def check_rows(windows, n_rows, rows_key):
    """The "recording", "start" and "length" columns of a windows dict checked on the host, as numpy int64: each a 1-D
    int64 tensor of n_rows rows (the row count of windows[rows_key]), recording and start >= 0, length >= 1, rows
    recording-major with start ascending and start + length non-decreasing within a recording.  Raises ValueError."""
    cols = []
    for k in ("recording", "start", "length"):
        v = windows[k]
        if not isinstance(v, torch.Tensor) or v.dim() != 1 or v.dtype != torch.int64:
            raise ValueError(f"{k} must be a 1-D int64 tensor")
        if v.numel() != n_rows:
            raise ValueError(f"{k} has {v.numel()} rows, {rows_key} {n_rows}")
        cols.append(v.cpu().numpy())
    rec, start, length = cols
    if (rec < 0).any() or (start < 0).any() or (length < 1).any():
        raise ValueError("recording and start must be >= 0 and length >= 1")
    if (np.diff(rec) < 0).any():
        raise ValueError("rows must be recording-major (recording non-decreasing)")
    same = np.diff(rec) == 0
    end = start + length
    if (np.diff(start)[same] <= 0).any() or (np.diff(end)[same] < 0).any():
        raise ValueError("within a recording, rows must have start ascending and start + length non-decreasing")
    return rec, start, length
