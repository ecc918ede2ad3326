"""CPU: the host side of sound event detection -- bin row ranges against brute-force intersection, the reference event
detector against an independent run-list implementation, the carried-state detector against the one-shot one, when a
stream emits each bin and event, a model of the row ring, validation, and the argument checks of the new entry points."""
import numpy as np
import pytest
import torch

import audioset_convnext_inf_b200 as acx
from audioset_convnext_inf_b200 import _native, sed
from audioset_convnext_inf_b200.engine import MIN_RAGGED_LEN
from audioset_convnext_inf_b200.stream import BinPlanner, StreamPlanner
from audioset_convnext_inf_b200.windows import plan_windows

W = 320000
C = 527


def _brute(starts, ends, n, R):
    """W_j by testing every window against every bin."""
    out = []
    for j in range(-(-n // R)):
        bs, be = j * R, min((j + 1) * R, n)
        out.append([i for i in range(len(starts)) if starts[i] < be and ends[i] > bs])
    return out


@pytest.mark.parametrize("hop", [32000, 99200, W])
@pytest.mark.parametrize("R", [32000, 16000, 45001, 10 ** 9])
def test_bin_ranges_equal_brute_force_intersection(hop, R):
    rng = np.random.default_rng(hop + R)
    lengths = [W, W - 1, W + 1, MIN_RAGGED_LEN, 3049600, 960017] + [int(x) for x in rng.integers(7360, 2_000_000, 4)]
    plan = plan_windows(lengths, W, hop)
    rec, start, length = (getattr(plan, k).numpy() for k in ("recording", "start", "length"))
    table, bins, seq = sed.plan_bins(rec, start, length, R)
    row = 0
    for r, n in enumerate(lengths):
        sel = np.flatnonzero(rec == r)
        ref = _brute(start[sel], start[sel] + length[sel], n, R)
        assert seq[r].tolist() == [r, row, len(ref), 0, n, 1]
        for j, rows in enumerate(ref):
            first, count, base, cap = table[row + j].tolist()
            assert list(range(first, first + count)) == [int(sel[0]) + i for i in rows] and rows, (r, j)
            assert (base, cap) == (0, len(rec))
            assert bins["recording"][row + j] == r and bins["start"][row + j] == j * R
            assert bins["length"][row + j] == min((j + 1) * R, n) - j * R
        row += len(ref)
    assert len(table) == row
    if R >= max(lengths):                                      # one bin per recording: all its windows
        assert table[:, 1].tolist() == [int((rec == r).sum()) for r in range(len(lengths))]


def test_hop_beyond_window_leaves_uncovered_bins():
    plan = plan_windows([2_000_000], 100000, 150000)
    args = [getattr(plan, k).numpy() for k in ("recording", "start", "length")]
    with pytest.raises(ValueError, match="covered by no window"):
        sed.plan_bins(*args, 32000)
    sed.plan_bins(*args, 10 ** 7)                              # one bin over everything is covered


# ---- events ---------------------------------------------------------------------------------------------------------------
def _runlist(a, starts, ends, on, off, gap, min_dur):
    """Independent run-list detector for one track: the hysteresis mask, its runs, then merging and the filter."""
    active = np.zeros(len(a), bool)
    for j in range(len(a)):
        active[j] = a[j] >= on or (j > 0 and active[j - 1] and a[j] >= off)
    runs, j = [], 0
    while j < len(a):
        if active[j]:
            k = j
            while k + 1 < len(a) and active[k + 1]:
                k += 1
            runs.append([starts[j], ends[k], float(np.max(a[j:k + 1]))])
            j = k + 1
        else:
            j += 1
    out = []
    for r in runs:
        if out and r[0] - out[-1][1] < gap:
            out[-1][1], out[-1][2] = r[1], max(out[-1][2], r[2])
        else:
            out.append(r)
    return [tuple(r) for r in out if r[1] - r[0] >= min_dur]


LEVELS = np.array([0.1, 0.3, 0.5, 0.7, np.nan], dtype=np.float32)     # off = 0.3 and on = 0.5 appear exactly


def _tracks(rng, n_bins, R, n=None):
    a = LEVELS[rng.integers(0, len(LEVELS), size=(n_bins, C))]
    a[rng.random((n_bins, C)) < 0.6] = np.float32(0.1)         # long quiet stretches: gaps of every size
    n = n_bins * R if n is None else n
    j = np.arange(n_bins, dtype=np.int64)
    return {"activity": a, "recording": np.zeros(n_bins, np.int64), "start": j * R,
            "length": np.minimum((j + 1) * R, n) - j * R}


@pytest.mark.parametrize("gap_bins, gap_extra", [(0, 0), (2, 0), (2, 1), (3, 0)])
@pytest.mark.parametrize("min_bins, min_extra", [(0, 0), (2, 0), (1, 500)])
def test_reference_events_equal_a_run_list_detector(gap_bins, gap_extra, min_bins, min_extra):
    R = 1000
    rng = np.random.default_rng(gap_bins * 10 + min_bins)
    act = _tracks(rng, 40, R, n=39 * R + 500)                    # a partial last bin of 500 samples
    on = np.full(C, 0.5, np.float32)
    off = np.full(C, 0.3, np.float32)
    on[::3], off[::3] = 0.7, 0.7                                  # per-class thresholds, on == off too
    off[1::3] = 0.1
    d = sed.Detection(R, on, off, min_duration_samples=min_bins * R + min_extra,
                      merge_gap_samples=gap_bins * R + gap_extra)
    got = sed.reference_events(act, d)
    starts, ends = act["start"], act["start"] + act["length"]
    want = []
    for c in range(C):
        want += [(0, c) + e for e in _runlist(act["activity"][:, c], starts, ends, on[c], off[c], d.merge_gap,
                                              d.min_duration)]
    assert len(got["onset"]) == len(want) > 0
    for i, (r, c, onset, offset, peak) in enumerate(want):
        assert (got["recording"][i], got["class"][i], got["onset"][i], got["offset"][i]) == (r, c, onset, offset)
        assert got["peak"][i] == np.float32(peak)
    if gap_extra:                                                 # a gap of exactly merge_gap - 1 samples merged ...
        merged = sed.reference_events(act, sed.Detection(R, on, off, 0, d.merge_gap))
        apart = sed.reference_events(act, sed.Detection(R, on, off, 0, gap_bins * R))
        assert len(merged["onset"]) < len(apart["onset"])          # ... a gap of exactly merge_gap is not
    ends_at_n = got["offset"] == 39 * R + 500
    assert ends_at_n.any()                                        # events that end in the partial bin


@pytest.mark.parametrize("seed", range(4))
def test_carried_state_in_random_splits_equals_one_shot(seed):
    rng = np.random.default_rng(seed)
    R = 1000
    nb = 60
    act = _tracks(rng, nb, R, n=(nb - 1) * R + 123)
    d = sed.Detection(R, 0.5, 0.3, min_duration_samples=int(rng.integers(0, 3)) * R,
                      merge_gap_samples=int(rng.integers(0, 4)) * R + int(rng.integers(0, 2)))
    ref = sed.reference_events(act, d)
    want = list(zip(ref["class"].tolist(), ref["onset"].tolist(), ref["offset"].tolist(), ref["peak"].tolist()))
    tracks = sed.EventTracks(d)
    cuts = sorted(set(rng.integers(0, nb - 1, size=6).tolist()) | {0})
    got = []
    for a, b in zip(cuts, cuts[1:]):                              # the partial last bin comes with close
        got += tracks.step(act["activity"][a:b], a, b * R, close=False)
    got += tracks.step(act["activity"][cuts[-1]:], cuts[-1], (nb - 1) * R + 123, close=True)
    got.sort(key=lambda e: (e[0], e[1]))
    assert [(c, o, f, np.float32(p)) for c, o, f, p in got] == [(c, o, f, np.float32(p)) for c, o, f, p in want]


# ---- streams --------------------------------------------------------------------------------------------------------------
def _chunks(rng, n):
    out, left = [], n
    while left > 0:
        m = min(left, (1, 32000, 700000, 0, int(rng.integers(1, 90000)))[int(rng.integers(5))])
        out.append(m)
        left -= m
    return out


@pytest.mark.parametrize("R, hop", [(32000, 32000), (16000, 99200), (45001, W), (10 ** 8, 32000)])
def test_stream_bins_final_on_time_and_ring_holds_every_row(R, hop):
    """Each bin is emitted by the first call after which it is final and never earlier; a model of the row ring (row
    ids instead of rows) shows every row a bin reads is held; the rows read are W_j of the whole stream's plan."""
    rng = np.random.default_rng(R + hop)
    rates = [32000, 44100, 32000, 48000]
    secs = [95.3, 41.0, 7.0, 0.4]                                # long, medium, shorter than a window, tiny
    lengths = [int(s * r) for s, r in zip(secs, rates)]
    lengths[3] = 11100                                           # 7400 samples at 32 kHz: one own-length window
    sp = StreamPlanner(rates, W, hop, piece_seconds=3)
    bp = BinPlanner(len(rates), W, hop, R, max(c - W for c in sp.out_cap))
    ring = np.full(len(rates) * bp.cap, -1, np.int64)
    chunked = [_chunks(rng, n) for n in lengths]
    n_calls = max(len(c) for c in chunked)
    emitted = {i: [] for i in range(len(rates))}                 # (bin, call)
    reads = {i: {} for i in range(len(rates))}
    k = [0] * len(rates)

    def piece(lengths_, close, t):
        pc = sp.step(lengths_, close)
        rec, start, length = (getattr(pc.plan, x).numpy() for x in ("recording", "start", "length"))
        slots, table, bins, seq = bp.step(rec, start, length, sp.n_final, close)
        for r, s in zip(rec.tolist(), slots.tolist()):
            ring[s] = (r << 32) | k[r]
            k[r] += 1
        for (first, count, base, cap), r, bs in zip(table.tolist(), bins["recording"].tolist(), bins["start"].tolist()):
            ids = [int(ring[base + (first + u) % cap]) for u in range(count)]
            assert ids == [(r << 32) | (first + u) for u in range(count)], ("row overwritten", r, bs)
            reads[r][bs // R] = list(range(first, first + count))
            emitted[r].append((bs // R, t))
        if seq is not None:
            assert seq[:, 2].sum() == len(table)

    for t in range(n_calls):
        push = [c[t] if t < len(c) else 0 for c in chunked]
        for pl in sp.split(push):
            piece(pl, (), t)
        for i in range(len(rates)):                              # not yet final: (j + 1) R > n_final - W
            done = [j for j, _ in emitted[i]]
            assert done == list(range(len(done)))
            assert len(done) == max(0, (sp.n_final[i] - W) // R), (i, t)
    piece([0] * len(rates), sp.check_close(None), n_calls)
    for i in range(len(rates)):
        n = sp.n_final[i]
        plan = plan_windows([n], W, hop)
        ref = _brute(plan.start.numpy(), (plan.start + plan.length).numpy(), n, R)
        assert [reads[i][j] for j in range(len(ref))] == ref and len(reads[i]) == len(ref)
        # emission timing: bin j in the first call after which (j + 1) R <= n_final - W, else at close
        fin = np.cumsum([0] + [c for c in chunked[i]])
        for j, t in emitted[i]:
            ok_at = [u for u in range(n_calls) if (j + 1) * R <= _final(sp, i, fin[min(u + 1, len(fin) - 1)]) - W]
            assert t == (ok_at[0] if ok_at else n_calls), (i, j, t)


def _final(sp, i, n_in):
    if sp.filt[i] is None:
        return n_in
    orig, new, width = sp.filt[i]
    return max(0, (n_in - width) // orig) * new


def test_stream_events_final_on_time():
    """EventTracks driven by the bins a stream makes final: each event comes from the first call after which no later
    bin can change it (the next bin starts merge_gap or more after its offset, or the stream closed), never earlier."""
    rng = np.random.default_rng(5)
    R = 1000
    nb = 80
    act = _tracks(rng, nb, R, n=(nb - 1) * R + 1)
    d = sed.Detection(R, 0.5, 0.3, min_duration_samples=R, merge_gap_samples=2 * R + 1)
    tr = sed.EventTracks(d)
    cuts = sorted(set(rng.integers(1, nb, size=12).tolist()))
    calls, done = [], 0
    for b in cuts + [nb]:
        close = b == nb
        limit = (nb - 1) * R + 1 if close else b * R
        calls.append((done, b, tr.step(act["activity"][done:b], done, limit, close)))
        done = b
    ref = sed.reference_events(act, d)
    allev = sorted(e for _, _, evs in calls for e in evs)
    assert [(c, o, f) for c, o, f, _ in allev] == sorted(zip(ref["class"].tolist(), ref["onset"].tolist(),
                                                              ref["offset"].tolist()))
    for t, (a, b, evs) in enumerate(calls):
        for c, onset, offset, _ in evs:
            final_now = b == nb or b * R - offset >= d.merge_gap
            final_before = a * R >= offset and a * R - offset >= d.merge_gap
            assert final_now and not final_before, (t, c, onset, offset)


def test_row_ring_size_does_not_depend_on_the_stream():
    bp = BinPlanner(3, W, 32000, 32000, 320000)
    assert bp.cap == (W + 32000 + 320000) // 32000 + 2
    with pytest.raises(ValueError, match="hop_samples <= window_samples"):
        BinPlanner(1, W, W + 1, 32000, 320000)


# ---- validation ---------------------------------------------------------------------------------------------------------
def test_detection_validation():
    for kw, msg in ((dict(resolution_samples=0), "resolution_samples"), (dict(resolution_samples=1.5), "resolution"),
                    (dict(resolution_samples=True), "resolution"), (dict(onset_threshold=float("nan")), "finite"),
                    (dict(onset_threshold=np.ones(526)), "shape"), (dict(offset_threshold=0.6), "exceeds"),
                    (dict(onset_threshold="0.5"), "dtype"), (dict(min_duration_samples=-1), "min_duration"),
                    (dict(merge_gap_samples=2.0), "merge_gap"), (dict(offset_threshold=np.inf), "finite")):
        args = dict(resolution_samples=32000, onset_threshold=0.5)
        args.update(kw)
        with pytest.raises(ValueError, match=msg):
            sed.Detection(**args)
    on = np.full(C, 0.5)
    off = on.copy()
    off[17] = 0.50001
    with pytest.raises(ValueError, match="class 17"):
        sed.Detection(32000, on, off)
    d = sed.Detection(32000, torch.full((C,), 0.5), None)
    assert d.on.dtype == np.float32 and (d.off == d.on).all()


def _windows(n_rows=5, **over):
    plan = plan_windows([W + 5 * 32000], W, 32000)
    w = {"clipwise_output": torch.rand(plan.start.numel(), C), "recording": plan.recording, "start": plan.start,
         "length": plan.length}
    w.update(over)
    return w


def test_detect_validates_rows_before_anything_else():
    d = sed.Detection(32000, 0.5)
    w = _windows()
    bad = [({"start": w["start"].flip(0)}, "start ascending"), ({"recording": torch.tensor([0, 0, 1, 0, 0, 0])},
                                                                  "recording-major"),
           ({"length": w["length"][:-1]}, "rows"), ({"start": w["start"].int()}, "int64"),
           ({"clipwise_output": w["clipwise_output"][:, :5]}, "527"), ({"length": w["length"] * 0}, "length >= 1"),
           ({"clipwise_output": w["clipwise_output"].double()}, "float32")]
    for over, msg in bad:
        with pytest.raises(ValueError, match=msg):
            sed.detect(_windows(**over), d)
    del w["start"]
    with pytest.raises(ValueError, match="lacks"):
        sed.detect(w, d)
    gaps = plan_windows([2_000_000], 100000, 150000)
    with pytest.raises(ValueError, match="covered by no window"):
        sed.detect({"clipwise_output": torch.rand(gaps.start.numel(), C), "recording": gaps.recording,
                    "start": gaps.start, "length": gaps.length}, d)
    with pytest.raises(ValueError, match="CUDA"):                 # every host check passes, then it needs the GPU
        sed.detect(_windows(), d)
    with pytest.raises(ValueError, match="Detection"):
        sed.detect(_windows(), {"resolution_samples": 32000})


def test_open_stream_validates_detection():
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56]).eval()
    with pytest.raises(ValueError, match="Detection"):
        m.open_stream(detection="dog")
    with pytest.raises(ValueError, match="hop_samples <= window_samples"):
        m.open_stream(hop_samples=W + 1, detection=sed.Detection(32000, 0.5))
    with pytest.raises(_native.NativeError):
        m.open_stream(detection=sed.Detection(32000, 0.5))


# ---- C ABI --------------------------------------------------------------------------------------------------------------
_P = 4096


def _activity_args(probs=_P, p_rows=100, table=_P, M=10, act=_P):
    return (probs, p_rows, table, M, act, 0)


def test_window_activity_entry_point_rejects_bad_arguments():
    fn = _native.load().acx_window_activity
    assert len(_native.SIGNATURES["acx_window_activity"]) == len(_activity_args())
    for kw in (dict(probs=0), dict(table=0), dict(act=0)):
        assert fn(*_activity_args(**kw)) == _native.ACX_ERR_ARG and "window_activity: null" in _native.last_error(), kw
    for kw, msg in ((dict(p_rows=0), "p_rows=0"), (dict(M=0), "M=0"), (dict(M=2 ** 40), "M=1099511627776")):
        assert fn(*_activity_args(**kw)) == _native.ACX_ERR_ARG and msg in _native.last_error(), kw
    assert fn(*([0] * len(_activity_args()))) == _native.ACX_ERR_ARG


def _events_args(act=_P, act_rows=10, seq=_P, S=2, on=_P, off=_P, R=32000, gap=0, min_dur=0, state=_P, peak=_P,
                 slots=_P, phase=0, out=_P, out_peak=_P, E=4):
    return (act, act_rows, seq, S, on, off, R, gap, min_dur, state, peak, slots, phase, out, out_peak, E, 0)


def test_detect_events_entry_point_rejects_bad_arguments():
    fn = _native.load().acx_detect_events
    assert len(_native.SIGNATURES["acx_detect_events"]) == len(_events_args())
    for kw in (dict(seq=0), dict(on=0), dict(off=0), dict(state=0), dict(peak=0), dict(slots=0), dict(act=0),
               dict(phase=1, out=0), dict(phase=1, out_peak=0)):
        assert fn(*_events_args(**kw)) == _native.ACX_ERR_ARG and "null" in _native.last_error(), kw
    for kw, msg in ((dict(S=0), "S=0"), (dict(S=2 ** 21), "S=2097152"), (dict(act_rows=-1), "act_rows=-1"),
                    (dict(E=-1), "E=-1"), (dict(R=0), "resolution 0"), (dict(gap=-1), "merge_gap -1"),
                    (dict(min_dur=-5), "min_duration -5"), (dict(phase=2), "bad phase 2"), (dict(phase=-1), "phase")):
        assert fn(*_events_args(**kw)) == _native.ACX_ERR_ARG and msg in _native.last_error(), kw
    assert fn(*([0] * len(_events_args()))) == _native.ACX_ERR_ARG
