"""Live streams: tag many audio streams window by window as their audio arrives (a bank of microphones, a call centre's
lines, broadcast channels).

ConvNeXt.open_stream returns a StreamTagger.  Each push appends every stream's new samples to a ring of its own on the
device and returns the windows that became complete; close ends streams and returns their last windows.  For every
stream, the rows of all calls together are exactly the rows forward_windows returns for the whole stream, bit for bit:
the windows are planned by plan_windows' rules and read in place by the same prep kernels (Engine.run_windows), and a
stream not at 32 kHz is resampled piece by piece with the same fmaf chain as preprocess.resample of the whole stream.

Device layout, fixed when the tagger is opened (one float32 buffer):
  output rings   stream i owns out_cap[i] + window slots at out_base[i].  Its 32 kHz sample t is written to slot
                 t mod out_cap[i] and, when that slot is below `window`, also to out_cap[i] + (t mod out_cap[i]) -- a
                 mirror of the ring's first `window` slots, so every window, one straddling the seam too, is contiguous
                 at out_base[i] + (start mod out_cap[i]) and the prep kernels read it as a window of a recording.
  input rings    a stream not at 32 kHz also owns in_cap[i] = K + piece input samples at in_base[i] (no mirror), K =
                 2 width + orig the taps of its reduced rate pair.  int16 chunks are converted x / 32767 on append.
Retention: the output ring holds the last `window` final samples plus one piece's new ones, which covers every regular
window still to come and the end-aligned tail; the input ring holds the last K input samples plus one piece, which
covers every input sample a not-yet-final output frame reads.  A push larger than one piece is run piece by piece.

Finality: output frame f of a resampled stream (outputs f*new .. f*new + new - 1) reads input samples
f*orig - width .. (f+1)*orig + width - 1, so it is final once (f+1)*orig + width <= n_in (input received so far).  At
close every frame up to ceil(total / new) is final, total = resampled_length(n_in, rate), and outputs past total are
not written.  A regular window [k hop, k hop + window) is returned by the call in which its last sample becomes final.

StreamPlanner is the pure-host part (counters, tables, window plans); StreamTagger owns the buffers and launches."""
import collections
import math
import numbers
import os

import numpy as np
import torch

from . import _native, preprocess, sed
from .engine import MIN_RAGGED_LEN, N_CLASSES, DIMS, out_time_dims
from .windows import WindowPlan, plan_windows

SAMPLE_RATE = preprocess.SAMPLE_RATE

# One piece of device work.  append: (A, 6) int64 rows (src_off, n, ring_base, cap, pos, mirror) of acx_stream_append,
# in stream order; resample: {rate: (R, 8) int64 rows (in_base, in_cap, in_end, f0, n_out, out_base, out_cap,
# out_mirror) of acx_resample_stream}; plan: windows.WindowPlan whose offsets are ring positions and whose recording /
# start are stream indices and stream positions (32 kHz samples).
Piece = collections.namedtuple("Piece", "append resample plan")


class StreamPlanner:
    """Host state of n streams: per stream the input received, the final 32 kHz output samples, the next regular window
    and whether it is closed; and the ring layout.  step() turns one piece into the tables of its launches and its
    window plan.  No device work happens here."""

    def __init__(self, rates, window=320000, hop=32000, piece_seconds=10):
        plan_windows([], window, hop)                      # plan_windows' own checks of window and hop
        if isinstance(piece_seconds, bool) or not isinstance(piece_seconds, numbers.Real) or not piece_seconds > 0 \
                or not math.isfinite(piece_seconds):
            raise ValueError(f"piece_seconds = {piece_seconds!r}: expected a positive number of seconds")
        self.window, self.hop = int(window), int(hop)
        self.rates = [int(r) for r in rates]
        S = len(self.rates)
        if S < 1:
            raise ValueError("a stream tagger needs at least one stream")
        self.piece_in = [max(1, int(piece_seconds * r)) for r in self.rates]   # input samples per stream and piece
        self.filt, self.out_cap, self.in_cap = [], [], []
        for r, m in zip(self.rates, self.piece_in):
            if r == SAMPLE_RATE:
                self.filt.append(None)
                self.out_cap.append(self.window + m)
                self.in_cap.append(0)
            else:
                orig, new, width = preprocess._rate_params(r, SAMPLE_RATE)
                self.filt.append((orig, new, width))
                # a piece of m inputs finalises at most m // orig + 1 frames; close at most width // orig + 3
                self.out_cap.append(self.window + max(m // orig + 1, width // orig + 3) * new)
                self.in_cap.append(2 * width + orig + m)
        regions = np.array([c + self.window for c in self.out_cap] + self.in_cap, dtype=np.int64)
        base = np.concatenate([[0], np.cumsum(regions)]).tolist()
        self.out_base = base[:S]
        self.in_base = base[S:2 * S]
        self.ring_len = base[-1]
        self.n_in = [0] * S            # input samples received
        self.n_final = [0] * S         # final 32 kHz output samples (a whole number of frames until close)
        self.next_k = [0] * S          # next regular window k: [k hop, k hop + window)
        self.closed = [False] * S

    @property
    def n_streams(self):
        return len(self.rates)

    def check_push(self, lengths):
        """lengths: one int per stream.  ValueError for a wrong count or new samples for a closed stream."""
        if len(lengths) != self.n_streams:
            raise ValueError(f"push got {len(lengths)} chunks for {self.n_streams} streams")
        for i, m in enumerate(lengths):
            if m and self.closed[i]:
                raise ValueError(f"stream {i} is closed: it takes no more samples")

    def check_close(self, streams=None):
        """The streams to close (None: every open one) as a sorted list.  ValueError for an unknown or closed stream, or
        one whose resampled length is shorter than the model takes (MIN_RAGGED_LEN samples)."""
        if streams is None:
            streams = [i for i in range(self.n_streams) if not self.closed[i]]
        elif isinstance(streams, numbers.Integral) and not isinstance(streams, bool):
            streams = [int(streams)]
        else:
            streams = list(streams)
        out = set()
        for i in streams:
            if isinstance(i, bool) or not isinstance(i, numbers.Integral) or not 0 <= int(i) < self.n_streams:
                raise ValueError(f"close: {i!r} is not a stream index in [0, {self.n_streams})")
            if self.closed[int(i)]:
                raise ValueError(f"close: stream {int(i)} is already closed")
            out.add(int(i))
        for i in sorted(out):
            n = preprocess.resampled_length(self.n_in[i], self.rates[i])
            if n < MIN_RAGGED_LEN:
                raise ValueError(f"stream {i} has {n} samples at 32 kHz; the shortest the model takes is {MIN_RAGGED_LEN}")
        return sorted(out)

    def split(self, lengths):
        """Per-piece chunk lengths of a push: piece p takes samples [p m_i, (p + 1) m_i) of stream i's chunk, m_i =
        piece_in[i].  No pieces for an empty push."""
        n = max([-(-int(x) // m) for x, m in zip(lengths, self.piece_in)] + [0])
        return [[min(m, max(0, int(x) - p * m)) for x, m in zip(lengths, self.piece_in)] for p in range(n)]

    def step(self, lengths, close=()):
        """Advance every stream by one piece (lengths[i] <= piece_in[i] new input samples) and close the streams in
        `close`; returns the Piece.  Arguments are assumed checked (check_push / check_close / split)."""
        close = set(close)
        W, hop = self.window, self.hop
        app, res = [], {}
        rec, start, length, offset = [], [], [], []
        src_off = 0
        for i in range(self.n_streams):
            m = int(lengths[i])
            filt = self.filt[i]
            if m:
                if filt is None:
                    app.append((src_off, m, self.out_base[i], self.out_cap[i], self.n_in[i] % self.out_cap[i], W))
                else:
                    app.append((src_off, m, self.in_base[i], self.in_cap[i], self.n_in[i] % self.in_cap[i], 0))
                src_off += m
            self.n_in[i] += m
            n_in = self.n_in[i]
            closing = i in close
            if filt is None:
                final = n_in
            else:
                orig, new, width = filt
                f0 = self.n_final[i] // new
                if closing:
                    final = preprocess.resampled_length(n_in, self.rates[i])
                else:
                    final = max(0, (n_in - width) // orig) * new
                if final > f0 * new:
                    res.setdefault(self.rates[i], []).append((self.in_base[i], self.in_cap[i], n_in, f0, final - f0 * new,
                                                             self.out_base[i], self.out_cap[i], W))
            self.n_final[i] = final
            starts = []
            k = self.next_k[i]
            while k * hop + W <= final:
                starts.append((k * hop, W))
                k += 1
            self.next_k[i] = k
            if closing:
                if final < W:
                    starts.append((0, final))              # a stream shorter than a window: one at its own length
                elif (k - 1) * hop + W < final:
                    starts.append((final - W, W))          # the end-aligned tail
                self.closed[i] = True
            for s, ln in starts:
                rec.append(i)
                start.append(s)
                length.append(ln)
                offset.append(self.out_base[i] + s % self.out_cap[i])

        def i64(v):
            return torch.tensor(v, dtype=torch.int64)

        plan = WindowPlan(i64(rec), i64(start), i64(length), i64(offset), W)
        return Piece(np.array(app, dtype=np.int64).reshape(-1, 6),
                     {r: np.array(rows, dtype=np.int64) for r, rows in res.items()}, plan)


class BinPlanner:
    """Host side of sound event detection on live streams (sed.py has the definitions): which activity bins became
    final, which window rows they read, and where those rows sit in the device row ring.  No device work happens here.

    Finality: while stream i is open, bin j is final iff (j + 1) R <= n_final_i - window.  No window still to come can
    then intersect it (a regular one starts at or after n_final - window + 1 and the end-aligned tail at n - window >=
    n_final - window), and every window that does is already complete.  At close every remaining bin is final.

    Row ring: stream i owns `cap` rows (rows i cap .. i cap + cap - 1 of one (S cap, 527) float32 buffer); its k-th window
    row goes to slot k mod cap.  A row is held until every bin it intersects is final, i.e. while start + window > j R
    for the first bin j not yet final, so the held rows start after n_final - 2 window - R; a piece adds rows starting up
    to n_final + piece_out - window, and close one end-aligned tail.  So cap = (window + R + piece_out) // hop + 2 rows
    (piece_out: the most 32 kHz samples one piece makes final) holds every row a not-yet-final bin reads.  hop > window
    leaves bins no window covers, so it is refused."""

    def __init__(self, n_streams, window, hop, resolution, piece_out):
        if hop > window:
            raise ValueError(f"detection needs hop_samples <= window_samples (got {hop} > {window}): with gaps between "
                             "windows some bins would be covered by no window")
        self.window, self.hop, self.R = int(window), int(hop), int(resolution)
        self.cap = (self.window + self.R + int(piece_out)) // self.hop + 2
        self.n_rows = [0] * n_streams         # window rows received: the next row's k
        self.first = [0] * n_streams          # k of the oldest held row
        self.starts = [np.zeros(0, np.int64) for _ in range(n_streams)]   # held rows' starts and ends
        self.ends = [np.zeros(0, np.int64) for _ in range(n_streams)]
        self.n_bins = [0] * n_streams         # final bins
        self.closed = [False] * n_streams

    def step(self, rec, start, length, n_final, close=()):
        """One piece: its window rows (recording = stream, start, length; stream-major), every stream's final 32 kHz
        samples after it, and the streams it closes.  Returns (slots (N,) int64 ring rows of the piece's rows, table
        (M, 4) int64 for acx_window_activity, bins {recording, start, length} (M,) int64, seq (S, 6) int64 for
        acx_detect_events or None when no bin became final and no stream closes)."""
        close = set(close)
        W, R, cap = self.window, self.R, self.cap
        slots = np.empty(len(rec), np.int64)
        for i in np.unique(rec).tolist():
            sel = np.flatnonzero(rec == i)
            slots[sel] = i * cap + (self.n_rows[i] + np.arange(sel.size)) % cap
            self.n_rows[i] += sel.size
            self.starts[i] = np.concatenate([self.starts[i], start[sel]])
            self.ends[i] = np.concatenate([self.ends[i], start[sel] + length[sel]])
            assert self.n_rows[i] - self.first[i] <= cap, "row ring bound violated"
        tables, b_rec, b_start, b_len, seq = [], [], [], [], []
        row0 = 0
        for i, n in enumerate(n_final):
            closing = i in close
            j0 = self.n_bins[i]
            total = -(-n // R) if closing else (j0 if self.closed[i] else max(j0, (n - W) // R))
            if total > j0:
                first, count = sed.bin_ranges(self.starts[i], self.ends[i], j0, total, R, n)
                assert (count >= 1).all(), "a final bin is covered by no window"
                tables.append(np.stack([self.first[i] + first, count, np.full_like(count, i * cap),
                                        np.full_like(count, cap)], axis=1))
                j = np.arange(j0, total, dtype=np.int64)
                b_rec.append(np.full(j.size, i, np.int64))
                b_start.append(j * R)
                b_len.append(np.minimum((j + 1) * R, n) - j * R)
                drop = int(np.searchsorted(self.ends[i], total * R, side="right"))   # no later bin reads these
                self.first[i] += drop
                self.starts[i], self.ends[i] = self.starts[i][drop:], self.ends[i][drop:]
            seq.append((i, row0, total - j0, j0, n if closing else total * R, int(closing)))
            row0 += total - j0
            self.n_bins[i] = total
            self.closed[i] |= closing

        def cat(parts, k=None):
            return np.concatenate(parts).astype(np.int64) if parts else np.zeros((0,) if k is None else (0, k), np.int64)

        bins = {"recording": cat(b_rec), "start": cat(b_start), "length": cat(b_len)}
        busy = row0 > 0 or bool(close)
        return slots, cat(tables, 4), bins, (np.array(seq, dtype=np.int64) if busy else None)


class StreamTagger:
    """n live streams tagged by one model (ConvNeXt.open_stream).  push() appends chunks and returns the windows that
    became complete; close() ends streams and returns their last windows.  See the module docstring for the layout.
    With a sed.Detection, every result also carries the activity bins and events that became final (BinPlanner)."""

    def __init__(self, model, n_streams=1, window_samples=320000, hop_samples=32000, sample_rate=32000,
                 frame_embeddings=False, piece_seconds=10, detection=None):
        model._check_inference(None)
        if isinstance(n_streams, bool) or not isinstance(n_streams, numbers.Integral) or n_streams < 1:
            raise ValueError(f"n_streams = {n_streams!r}: expected a positive int")
        rates = preprocess.sample_rates(sample_rate, int(n_streams))
        self.planner = StreamPlanner(rates, window_samples, hop_samples, piece_seconds)
        self.detection = detection
        if detection is not None:
            if not isinstance(detection, sed.Detection):
                raise ValueError("detection must be a sed.Detection or None")
            p = self.planner
            self.bins = BinPlanner(p.n_streams, p.window, p.hop, detection.resolution,
                                   max(c - p.window for c in p.out_cap))
        self.model = model
        self.frame_embeddings = bool(frame_embeddings)
        eng = model._get_engine()
        self.device = eng.device
        self._filters = {}
        for r in sorted(set(rates) - {SAMPLE_RATE}):
            taps, width, orig, new = preprocess._cached_taps(r, SAMPLE_RATE, self.device)
            self._filters[r] = (taps, width, orig, new) + preprocess.segment_tiling(orig, new, width)
        # NaN until written: a read of a slot no sample has reached shows in the results
        self.ring = torch.full((self.planner.ring_len,), float("nan"), dtype=torch.float32, device=self.device)
        if detection is not None:
            self.row_ring = torch.full((self.planner.n_streams * self.bins.cap, N_CLASSES), float("nan"),
                                       dtype=torch.float32, device=self.device)
            self.sed_state = sed.new_state(self.planner.n_streams, self.device)

    @property
    def ring_bytes(self):
        return self.ring.numel() * self.ring.element_size()

    @property
    def detection_bytes(self):
        """Device memory of detection, fixed at open: the row ring (BinPlanner.cap rows of 527 float32 per stream) and
        the per-track event state (3 int64 + 1 float32 per stream and class); 0 without detection."""
        if self.detection is None:
            return 0
        return sum(t.numel() * t.element_size() for t in (self.row_ring,) + self.sed_state)

    def _chunks(self, chunks):
        S = self.planner.n_streams
        if chunks is None or isinstance(chunks, (torch.Tensor, np.ndarray)):
            if S != 1:
                raise ValueError(f"push got one chunk for {S} streams: pass a sequence of {S} chunks (None for none)")
            chunks = [chunks]
        chunks = list(chunks)
        if len(chunks) != S:
            raise ValueError(f"push got {len(chunks)} chunks for {S} streams")
        out = []
        for i, c in enumerate(chunks):
            if c is None:
                out.append(None)
                continue
            c = c if isinstance(c, torch.Tensor) else torch.as_tensor(c)
            if c.dim() != 1:
                raise ValueError(f"chunk {i} must be 1-D (samples), got shape {tuple(c.shape)}")
            if not (c.dtype == torch.int16 or c.is_floating_point()):
                raise ValueError(f"chunk {i} has dtype {c.dtype}: expected a float dtype or int16 PCM")
            out.append(c.detach() if c.numel() else None)
        return out

    def push(self, chunks):
        """Append new samples: one 1-D tensor (n_streams == 1) or a sequence of n_streams entries, each a 1-D tensor or
        array on the host or the device (float32, int16 PCM read x / 32767, or another float dtype) of any length, or
        None / empty for nothing new.  Returns the rows of the windows that became complete (see ConvNeXt.open_stream).
        Every argument is checked before anything is copied or launched."""
        self.model._check_inference(None)
        chunks = self._chunks(chunks)
        lengths = [0 if c is None else c.numel() for c in chunks]
        self.planner.check_push(lengths)
        parts = []
        done = [0] * len(chunks)
        for piece_lengths in self.planner.split(lengths):
            sub = [chunks[i][done[i]:done[i] + m] for i, m in enumerate(piece_lengths) if m]
            for i, m in enumerate(piece_lengths):
                done[i] += m
            parts.append(self._piece(piece_lengths, sub, ()))
        return self._gather(parts)

    def close(self, streams=None):
        """End `streams` (one index, a sequence of indices, or None for every open stream) and return their last rows:
        the windows that became final at the end of the stream, the end-aligned tail window, and for a stream shorter
        than a window its one own-length window.  A stream whose resampled length is under 7360 samples raises
        ValueError before anything is launched, and no stream is closed."""
        self.model._check_inference(None)
        streams = self.planner.check_close(streams)
        if not streams:
            return self._gather([])
        return self._gather([self._piece([0] * self.planner.n_streams, [], streams)])

    @property
    def closed(self):
        return list(self.planner.closed)

    # ---- device work of one piece ------------------------------------------------------------------------------------
    def _pack(self, sub):
        """The piece's chunks end to end on the device (int16 when every one is int16, else float32) with one copy."""
        if all(not c.is_cuda for c in sub):
            host = preprocess.pack_waveforms(sub, torch.device("cpu"), pin_memory=True)
            own = len(sub) == 1 and host.data_ptr() == sub[0].data_ptr()     # pack_waveforms made no copy
            if not host.is_pinned():
                host, own = host.pin_memory(), False
            # a caller's own pinned tensor may be refilled as soon as push returns: copy it synchronously
            return host.to(self.device, non_blocking=not own)
        return preprocess.pack_waveforms(sub, self.device)

    def _piece(self, lengths, sub, close):
        eng = self.model._get_engine()
        dev = self.device
        x = self._pack(sub) if sub else None
        old_final = list(self.planner.n_final)
        piece = self.planner.step(lengths, close)
        st = torch.cuda.current_stream(dev).cuda_stream
        ring = self.ring
        if len(piece.append):
            tab = torch.from_numpy(piece.append).pin_memory().to(dev, non_blocking=True)
            entry = "acx_stream_append_pcm16" if x.dtype == torch.int16 else "acx_stream_append"
            _native.call(entry, x.data_ptr(), x.numel(), tab.data_ptr(), len(piece.append), ring.data_ptr(), ring.numel(),
                         st)
        for r, rows in piece.resample.items():
            taps, width, orig, new, tile_frames, phase_groups = self._filters[r]
            start, n_tiles = preprocess.segment_tiles(rows[:, 4].tolist(), tile_frames, phase_groups, new)
            S = len(rows)
            table = torch.cat([torch.from_numpy(rows).flatten(), start]).pin_memory().to(dev, non_blocking=True)
            _native.call("acx_resample_stream", ring.data_ptr(), ring.numel(), table.data_ptr(), S,
                         table.data_ptr() + 8 * 8 * S, n_tiles, taps.data_ptr(), orig, new, width, ring.data_ptr(),
                         ring.numel(), st)
        self._check_amplitude(eng, old_final)
        plan = piece.plan
        res = None
        if plan.length.numel():
            want = ("logits", "scene", "frame") if self.frame_embeddings else ("logits", "scene")
            out = eng.run_windows(ring, plan, want)
            res = {"clipwise_output": out["probs"], "clipwise_logits": out["logits"], "scene_embeddings": out["scene"],
                   "recording": plan.recording, "start": plan.start, "length": plan.length}
            if self.frame_embeddings:
                res["frame_embeddings"] = out["frame"]
        return res, (self._detect(plan, res, close) if self.detection is not None else None)

    def _detect(self, plan, res, close):
        """The piece's rows into the row ring, then the bins that became final and the events they finalise."""
        slots, table, bins, seq = self.bins.step(plan.recording.numpy(), plan.start.numpy(), plan.length.numpy(),
                                                 self.planner.n_final, close)
        if len(slots):
            idx = torch.from_numpy(slots).pin_memory().to(self.device, non_blocking=True)
            self.row_ring.index_copy_(0, idx, res["clipwise_output"])
        act = sed.window_activity(self.row_ring, table)
        events = sed.detect_events(act, seq, self.detection, self.sed_state) if seq is not None else None
        return act, bins, events

    def _check_amplitude(self, eng, old_final):
        """ACX_CHECK_AMPLITUDE=1: the 32 kHz samples that became final in this piece (resampled where the stream is not at
        32 kHz) are checked as forward_windows checks its recording buffer, before any window reads them."""
        if os.environ.get("ACX_CHECK_AMPLITUDE") != "1" or eng.precision != "bf16":
            return
        p = self.planner
        parts = []
        for i, (a, b) in enumerate(zip(old_final, p.n_final)):
            while a < b:                                   # at most two contiguous runs of the ring per stream
                s = a % p.out_cap[i]
                m = min(b - a, p.out_cap[i] - s)
                parts.append(self.ring[p.out_base[i] + s:p.out_base[i] + s + m].abs().amax())
                a += m
        if parts:
            self.model._check_amplitude(eng, torch.stack(parts))

    def _gather(self, parts):
        """The rows of all pieces of one call, stream-major with start ascending, on the device; with detection also its
        activity bins (stream-major, start ascending) and events (stream, class, onset)."""
        res = self._gather_rows([p[0] for p in parts if p[0] is not None])
        if self.detection is not None:
            res["activity"], res["events"] = self._gather_sed([p[1] for p in parts])
        return res

    def _gather_sed(self, parts):
        dev = self.device
        host = {k: np.concatenate([p[1][k] for p in parts] + [np.zeros(0, np.int64)]) for k in sed.ACTIVITY_KEYS[1:]}
        acts = [p[0] for p in parts if len(p[0])]
        act = torch.cat(acts) if acts else torch.empty(0, N_CLASSES, dtype=torch.float32, device=dev)
        if len(acts) > 1:                 # pieces come in time order: a stable sort on the stream keeps start ascending
            order = np.argsort(host["recording"], kind="stable")
            host = {k: v[order] for k, v in host.items()}
            act = act.index_select(0, torch.from_numpy(order).to(dev, non_blocking=True))
        activity = {"activity": act}
        activity.update({k: torch.from_numpy(v).to(dev) for k, v in host.items()})
        evs = [p[2] for p in parts if p[2] is not None and p[2]["onset"].numel()]
        if not evs:
            empty = torch.zeros(0, dtype=torch.int64, device=dev)
            events = {k: empty for k in sed.EVENT_KEYS[:-1]}
            events["peak"] = torch.empty(0, dtype=torch.float32, device=dev)
        else:
            events = {k: torch.cat([e[k] for e in evs]) for k in sed.EVENT_KEYS}
            if len(evs) > 1:              # a track's events come in onset order, piece after piece
                order = torch.sort(events["recording"] * N_CLASSES + events["class"], stable=True).indices
                events = {k: v.index_select(0, order) for k, v in events.items()}
        return activity, events

    def _gather_rows(self, parts):
        dev = self.device
        h3w = out_time_dims(self.planner.window)[1][3]
        if not parts:
            f32 = dict(device=dev, dtype=torch.float32)
            res = {"clipwise_output": torch.empty(0, N_CLASSES, **f32), "clipwise_logits": torch.empty(0, N_CLASSES, **f32),
                   "scene_embeddings": torch.empty(0, DIMS[3], **f32)}
            host = {k: torch.zeros(0, dtype=torch.int64) for k in ("recording", "start", "length")}
            if self.frame_embeddings:
                res["frame_embeddings"] = torch.empty(0, DIMS[3], h3w, 7, **f32)
        elif len(parts) == 1:
            res = {k: v for k, v in parts[0].items() if k not in ("recording", "start", "length")}
            host = {k: parts[0][k] for k in ("recording", "start", "length")}
        else:
            host = {k: torch.cat([p[k] for p in parts]) for k in ("recording", "start", "length")}
            # pieces come in time order, so a stable sort on the stream index keeps each stream's starts ascending
            order = torch.from_numpy(np.argsort(host["recording"].numpy(), kind="stable"))
            host = {k: v[order] for k, v in host.items()}
            idx = order.to(dev, non_blocking=True)
            res = {k: torch.cat([p[k] for p in parts]).index_select(0, idx) for k in parts[0]
                   if k not in ("recording", "start", "length")}
        for k, v in host.items():
            res[k] = v.to(dev)
        if self.frame_embeddings:
            h3 = [out_time_dims(n)[1][3] for n in host["length"].tolist()]
            res["frame_lengths"] = torch.tensor(h3, dtype=torch.int64).to(dev)
        return res
