"""CPU: the host side of live streams -- StreamPlanner against plan_windows over random chunkings, when each window and
each resampled frame is emitted, a model of the append and resample kernels' ring index arithmetic (sample ids instead
of samples), validation before any device work, and the argument checks of the new entry points."""
import numpy as np
import pytest

import audioset_convnext_inf_b200 as acx
from audioset_convnext_inf_b200 import _native
from audioset_convnext_inf_b200.engine import MIN_RAGGED_LEN
from audioset_convnext_inf_b200.preprocess import _rate_params, resampled_length
from audioset_convnext_inf_b200.stream import StreamPlanner
from audioset_convnext_inf_b200.windows import plan_windows

W = 320000
HOPS = (32000, 100001, 400000)


def _chunking(rng, n, piece):
    """Chunk sizes summing to n: 1-sample chunks, exactly a hop, far more than a piece, empty pushes, random."""
    sizes, left = [], n
    while left > 0:
        kind = rng.integers(6)
        m = (1, 32000, 3 * piece + int(rng.integers(piece)), 0, int(rng.integers(1, 50000)), int(rng.integers(1, 400000)))[kind]
        m = min(m, left)
        sizes.append(m)
        left -= m
    return sizes


def _drive(planner, pushes):
    """What StreamTagger.push / close do on the host: each push split into pieces, one step per piece.  Returns per
    call [(recording, start, length)] and the pieces of every call."""
    calls = []
    for lengths in pushes:
        planner.check_push(lengths)
        pieces = [planner.step(p) for p in planner.split(lengths)]
        calls.append(pieces)
    close = planner.check_close(None)
    calls.append([planner.step([0] * planner.n_streams, close)])
    return calls


def _rows(pieces):
    out = []
    for pc in pieces:
        out += list(zip(pc.plan.recording.tolist(), pc.plan.start.tolist(), pc.plan.length.tolist()))
    return out


def _final(planner, i, n_in):
    """Final 32 kHz samples of stream i after n_in input samples (before close)."""
    if planner.filt[i] is None:
        return n_in
    orig, new, width = planner.filt[i]
    return max(0, (n_in - width) // orig) * new


@pytest.mark.parametrize("hop", HOPS)
@pytest.mark.parametrize("rate", [32000, 44100])
def test_planner_equals_plan_windows_and_emits_on_time(hop, rate):
    rng = np.random.default_rng(hop + rate)
    lengths = [W, W - 1, W + 1, MIN_RAGGED_LEN, 3049600, 960017, 240000, 1234567]
    if rate != 32000:
        lengths = [n * rate // 32000 + 3 for n in lengths]
    for trial in range(3):
        p = StreamPlanner([rate] * len(lengths), W, hop, piece_seconds=(10, 1, 0.37)[trial])
        chunkings = [_chunking(rng, n, p.piece_in[i]) for i, n in enumerate(lengths)]
        n_calls = max(len(c) for c in chunkings)
        pushes = [[c[t] if t < len(c) else 0 for c in chunkings] for t in range(n_calls)]
        calls = _drive(p, pushes)
        got = {i: [] for i in range(len(lengths))}
        received = [0] * len(lengths)
        for t, pieces in enumerate(calls):
            for pc in pieces:                                     # each piece's plan is stream-major
                assert pc.plan.recording.tolist() == sorted(pc.plan.recording.tolist())
            for r, s, ln in _rows(pieces):
                got[r].append((s, ln))
            if t < len(pushes):
                for i in range(len(lengths)):
                    received[i] += pushes[t][i]
                    fin = _final(p, i, received[i])
                    # every regular window complete by now was emitted, none that is not (emission timing)
                    regular = [(s, W) for s in range(0, fin - W + 1, hop)]
                    assert got[i] == regular, (i, t)
        for i, n in enumerate(lengths):
            ref = plan_windows([resampled_length(n, rate)], W, hop)
            assert got[i] == list(zip(ref.start.tolist(), ref.length.tolist())), (i, n)
        assert all(p.closed)


def test_short_stream_at_close_raises_and_changes_nothing():
    p = StreamPlanner([32000, 44100], W, 32000)
    p.step([MIN_RAGGED_LEN - 1, 50000])
    state = (list(p.n_in), list(p.n_final), list(p.next_k), list(p.closed))
    with pytest.raises(ValueError, match="stream 0 has 7359 samples"):
        p.check_close(None)
    with pytest.raises(ValueError, match="stream 0"):
        p.check_close([1, 0])
    assert (p.n_in, p.n_final, p.next_k, p.closed) == state
    assert p.check_close(1) == [1]
    p.step([0, 0], [1])
    with pytest.raises(ValueError, match="closed"):
        p.check_push([5, 5])
    p.check_push([5, 0])                                          # nothing new for a closed stream is fine
    with pytest.raises(ValueError, match="already closed"):
        p.check_close([1])
    with pytest.raises(ValueError, match="2 streams"):
        p.check_push([5])
    for bad in ([2], [-1], [True], ["0"]):
        with pytest.raises(ValueError, match="stream index"):
            p.check_close(bad)


@pytest.mark.parametrize("rate", [44100, 48000, 8000, 22050])
def test_resampled_frames_are_final_exactly_when_their_input_is(rate):
    rng = np.random.default_rng(rate)
    orig, new, width = _rate_params(rate, 32000)
    for n in (rate * 7 + 13, 2 * orig + 5, rate // 3):
        p = StreamPlanner([rate], W, 32000, piece_seconds=0.5)
        sizes = _chunking(rng, n, p.piece_in[0])
        received, frames, emitted_at = 0, [], {}
        for t, m in enumerate(sizes):
            for lengths in p.split([m]):
                pc = p.step(lengths)
                for row in pc.resample.get(rate, []):
                    f0, n_out = int(row[3]), int(row[4])
                    assert n_out % new == 0                        # whole frames until close
                    for f in range(f0, f0 + n_out // new):
                        emitted_at[f] = t
                        frames.append(f)
                    assert row[2] == p.n_in[0]                    # in_end: everything received so far
            received += m
        last = sum(1 for _ in sizes)
        pc = p.step([0], [0])
        total = resampled_length(n, rate)
        for row in pc.resample.get(rate, []):
            f0, n_out = int(row[3]), int(row[4])
            assert f0 * new + n_out == total                      # outputs past the stream's length are not computed
            for f in range(f0, -(-total // new)):
                emitted_at[f] = last
                frames.append(f)
        assert frames == list(range(-(-total // new)))            # each frame once, in order
        assert p.n_final[0] == total
        cum = np.cumsum(sizes)
        for f, t in emitted_at.items():
            first = next((u for u, c in enumerate(cum) if (f + 1) * orig + width <= c), last)
            assert t == first, (f, t, first)


# ---- a model of the kernels' index arithmetic --------------------------------------------------------------------------
def _ident(s, t):
    return (np.int64(s) << 40) | np.asarray(t, dtype=np.int64)


def _append(ring, app, src_ids):
    """stream_append_kernel: chunk row (src_off, n, base, cap, pos, mirror) -> slot (pos + i) mod cap, mirrored."""
    for src_off, n, base, cap, pos, mirror in app.tolist():
        n = min(max(n, 0), cap)
        i = np.arange(n)
        slot = pos + i
        slot = np.where(slot >= cap, slot - cap, slot)
        assert (slot < cap).all()                                 # pos < cap: the kernel's one-subtraction path
        ring[base + slot] = src_ids[src_off:src_off + n]
        m = slot < mirror
        ring[base + cap + slot[m]] = src_ids[src_off:src_off + n][m]


def _resample(ring, rows, orig, new, width, stream_of):
    """resample_segments_kernel<float, true>: checks every frame's input span, then writes the output ids."""
    K = 2 * width + orig
    for in_base, in_cap, in_end, f0, n_out, out_base, out_cap, mirror in rows.tolist():
        s = stream_of[out_base]
        for f in range(f0, f0 + -(-n_out // new)):
            idx = f * orig - width + np.arange(K)
            live = (idx >= 0) & (idx < in_end)
            seen = ring[in_base + np.mod(idx[live], in_cap)]
            assert (seen == _ident(s, idx[live])).all(), ("stale or overwritten input", s, f)
        j = f0 * new + np.arange(n_out)
        slot = np.mod(j, out_cap)
        ring[out_base + slot] = _ident(s, j)
        m = slot < mirror
        ring[out_base + out_cap + slot[m]] = _ident(s, j[m])


@pytest.mark.parametrize("hop", HOPS)
def test_ring_simulation_every_window_and_frame_reads_the_right_samples(hop):
    rates = [32000, 44100, 8000, 48000, 32000]
    window = 96000                                                # 3 s windows so that the rings wrap many times
    p = StreamPlanner(rates, window, hop, piece_seconds=0.3)
    filt = {r: _rate_params(r, 32000) for r in set(rates) if r != 32000}
    stream_of = {b: i for i, b in enumerate(p.out_base)}
    ring = np.full(p.ring_len, -1, dtype=np.int64)
    rng = np.random.default_rng(hop)
    secs = [41.3, 17.01, 23.5, 2.2, 0.9]
    lengths = [int(s * r) for s, r in zip(secs, rates)]
    chunkings = [_chunking(rng, n, p.piece_in[i]) for i, n in enumerate(lengths)]
    n_calls = max(len(c) for c in chunkings)
    pushes = [[c[t] if t < len(c) else 0 for c in chunkings] for t in range(n_calls)]
    received = [0] * len(rates)
    seam = 0
    windows = 0

    def run(pc, lengths):
        nonlocal seam, windows
        src = np.concatenate([_ident(i, np.arange(received[i], received[i] + m)) for i, m in enumerate(lengths) if m]
                             + [np.zeros(0, np.int64)])
        for i, m in enumerate(lengths):
            received[i] += m
        _append(ring, pc.append, src)
        for r, rows in pc.resample.items():
            _resample(ring, rows, *filt[r], stream_of)
        for r, s, ln, off in zip(*(getattr(pc.plan, k).tolist() for k in ("recording", "start", "length", "offset"))):
            assert (ring[off:off + ln] == _ident(r, np.arange(s, s + ln))).all(), ("window reads wrong samples", r, s)
            seam += (s % p.out_cap[r]) + ln > p.out_cap[r]
            windows += 1

    for lengths in pushes:
        for pl in p.split(lengths):
            run(p.step(pl), pl)
    close = p.check_close(None)
    run(p.step([0] * len(rates), close), [0] * len(rates))
    assert seam > 0 and windows > 0
    for i in range(len(rates)):
        assert p.n_final[i] // p.out_cap[i] >= (3 if secs[i] > 10 else 0)   # long streams wrapped their ring many times


def test_ring_layout_and_memory_do_not_depend_on_the_stream():
    p = StreamPlanner([32000, 44100], W, 32000, piece_seconds=10)
    orig, new, width = _rate_params(44100, 32000)
    assert p.out_cap == [W + 320000, W + (441000 // orig + 1) * new]
    assert p.in_cap == [0, 2 * width + orig + 441000]
    assert p.out_base == [0, p.out_cap[0] + W]
    assert p.in_base[1] == p.out_base[1] + p.out_cap[1] + W
    assert p.ring_len == p.in_base[1] + p.in_cap[1]
    before = p.ring_len
    for _ in range(30):
        p.step([320000, 441000])
    assert p.ring_len == before


def test_open_stream_validates_before_touching_a_device():
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56]).eval()
    for kw, msg in ((dict(n_streams=0), "n_streams"), (dict(n_streams=2.0), "n_streams"),
                    (dict(sample_rate=0), "sample_rate"), (dict(n_streams=2, sample_rate=[44100]), "sample_rate"),
                    (dict(window_samples=7359), "window_samples"), (dict(hop_samples=0), "hop_samples"),
                    (dict(piece_seconds=0), "piece_seconds"), (dict(piece_seconds=float("inf")), "piece_seconds")):
        with pytest.raises(ValueError, match=msg):
            m.open_stream(**kw)
    with pytest.raises(_native.NativeError):                      # every check passes, then it needs the GPU
        m.open_stream(n_streams=2, sample_rate=[44100, 32000])
    m.train()
    with pytest.raises(RuntimeError, match="eval"):
        m.open_stream()


# ---- C ABI: the new entry points check their arguments before they touch a device ---------------------------------------
_P = 4096        # a non-null dummy address: the calls below must fail before dereferencing anything


def _append_args(src=_P, src_len=1000, tab=_P, S=2, ring=_P, ring_len=10 ** 6):
    return (src, src_len, tab, S, ring, ring_len, 0)


@pytest.mark.parametrize("name", ["acx_stream_append", "acx_stream_append_pcm16"])
def test_append_entry_points_reject_bad_arguments(name):
    fn = getattr(_native.load(), name)
    assert len(_native.SIGNATURES[name]) == len(_append_args())
    for kw in (dict(src=0), dict(tab=0), dict(ring=0)):
        assert fn(*_append_args(**kw)) == _native.ACX_ERR_ARG and "null" in _native.last_error(), kw
    for kw, msg in ((dict(S=0), "S=0"), (dict(S=-3), "S=-3"), (dict(src_len=0), "src_len=0"),
                    (dict(src_len=2 ** 40), "src_len=1099511627776"), (dict(ring_len=0), "ring_len=0")):
        assert fn(*_append_args(**kw)) == _native.ACX_ERR_ARG and msg in _native.last_error(), kw
    assert fn(*([0] * len(_append_args()))) == _native.ACX_ERR_ARG


def _stream_args(x=_P, x_len=10 ** 6, tab=_P, S=2, tiles=_P, n_tiles=100, taps=_P, orig=441, new=320, width=9, out=_P,
                 out_len=10 ** 6):
    return (x, x_len, tab, S, tiles, n_tiles, taps, orig, new, width, out, out_len, 0)


def test_resample_stream_entry_point_rejects_bad_arguments():
    fn = _native.load().acx_resample_stream
    assert len(_native.SIGNATURES["acx_resample_stream"]) == len(_stream_args())
    for kw in (dict(x=0), dict(tab=0), dict(tiles=0), dict(taps=0), dict(out=0)):
        assert fn(*_stream_args(**kw)) == _native.ACX_ERR_ARG and "resample_stream: null" in _native.last_error(), kw
    for kw, msg in ((dict(S=0), "S=0"), (dict(x_len=0), "x_len=0"), (dict(out_len=-1), "out_len=-1"),
                    (dict(n_tiles=0), "n_tiles=0"), (dict(n_tiles=2 ** 31), "n_tiles"), (dict(orig=0), "rates"),
                    (dict(new=-320), "rates"), (dict(width=0), "width 0")):
        assert fn(*_stream_args(**kw)) == _native.ACX_ERR_ARG and msg in _native.last_error(), kw
    assert fn(*_stream_args(orig=5507, new=4000, width=9)) == _native.ACX_ERR_UNSUPPORTED
    assert fn(*([0] * len(_stream_args()))) == _native.ACX_ERR_ARG
