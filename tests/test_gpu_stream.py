"""GPU (B200): live streams -- ConvNeXt.open_stream.

For every stream, the rows of all push / close calls together must equal forward_windows of the whole stream, BIT FOR
BIT, for every key, however the stream is cut into chunks; resampled streams must equal forward_windows(...,
sample_rate=...).  The rings are NaN-filled when the tagger is opened, so a read of a slot no sample has reached shows
up as a mismatch."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import audioset_convnext_inf_b200 as acx                         # noqa: E402
from audioset_convnext_inf_b200 import _native, preprocess       # noqa: E402
from audioset_convnext_inf_b200.stream import StreamPlanner      # noqa: E402

DEV = "cuda:0"
W = 320000
KEYS = ("clipwise_output", "clipwise_logits", "scene_embeddings", "start", "length", "frame_embeddings", "frame_lengths")
# 95.3 s (end-aligned tail), exactly 10 s, 7.5 s (one window at its own length), 30 s + 17 samples
LENGTHS = (3049600, W, 240000, 960017)


def _model(sd, prec):
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval().set_precision(prec)


@pytest.fixture(scope="module")
def models(parity_sd):
    return {prec: _model(parity_sd, prec) for prec in ("fp32", "bf16")}


def _signal(n, rng, pcm=False):
    if pcm:
        return torch.from_numpy(rng.integers(-6000, 6000, size=n).astype(np.int16))
    return torch.from_numpy(np.clip(rng.standard_normal(n) * 0.1, -1, 1).astype(np.float32))


def _cut(rec, rng, piece):
    """rec cut into chunks: 1-sample chunks, exactly a hop, far more than a piece, random sizes."""
    out, at = [], 0
    while at < rec.numel():
        m = (1, 32000, 2 * piece + int(rng.integers(piece)), int(rng.integers(1, 60000)), int(rng.integers(1, 500000)))[
            int(rng.integers(5))]
        out.append(rec[at:at + m])
        at += m
    return out


def _as_float(c):
    return preprocess.pack_waveforms([c], torch.device("cpu")) if c.dtype == torch.int16 else c.to(torch.float32)


def _run(s, streams, rng, close_after=None, device_every=3):
    """Push every stream's chunks (None once a stream has none left, and now and then for all), closing stream i after
    push close_after[i].  Returns the rows of all calls."""
    n_calls = max(len(c) for c in streams)
    calls = []
    for t in range(n_calls):
        push = []
        for i, cs in enumerate(streams):
            c = cs[t] if t < len(cs) else None
            if c is not None and t % device_every == 1:
                c = c.to(DEV)
            elif c is not None and t % 7 == 3 and c.is_floating_point():
                c = c.double()                                     # any float dtype is cast to float32
            if s.closed[i]:
                c = None
            push.append(c)
        calls.append(s.push(push))
        if close_after:
            due = [i for i, t_i in close_after.items() if t_i == t]
            if due:
                calls.append(s.close(due))
    if not all(s.closed):
        calls.append(s.close())
    return calls


def _stream_rows(calls, i):
    out = {}
    for k in calls[0]:
        rows = [c[k][c["recording"] == i] for c in calls]
        out[k] = torch.cat(rows)
    return out


def _assert_equal(got, ref, what):
    for k in KEYS:
        if k in ref:
            assert got[k].dtype == ref[k].dtype and got[k].device == ref[k].device, (what, k)
            assert torch.equal(got[k], ref[k]), (what, k)


def _check_calls(calls, n_streams):
    for c in calls:
        rec = c["recording"].tolist()
        assert rec == sorted(rec)                                  # stream-major ...
        for i in set(rec):
            st = c["start"][c["recording"] == i].tolist()
            assert st == sorted(st)                                # ... start ascending
    assert {r for c in calls for r in c["recording"].tolist()} <= set(range(n_streams))


@pytest.mark.parametrize("prec, hop", [("bf16", 32000), ("bf16", 100001), ("bf16", 400000), ("fp32", 100001)])
def test_rows_bit_identical_to_forward_windows_of_the_whole_stream(models, prec, hop):
    m = models[prec]
    rng = np.random.default_rng(hop)
    recs = [_signal(n, rng) for n in LENGTHS]
    s = m.open_stream(len(recs), W, hop, frame_embeddings=True)
    assert torch.isnan(s.ring).all()                               # poison: unwritten slots are NaN
    piece = s.planner.piece_in[0]
    with torch.no_grad():
        calls = _run(s, [_cut(r, rng, piece) for r in recs], rng)
        _check_calls(calls, len(recs))
        seam = 0
        for i, rec in enumerate(recs):
            got = _stream_rows(calls, i)
            ref = m.forward_windows(rec, W, hop, frame_embeddings=True)
            _assert_equal(got, ref, i)
            cap = s.planner.out_cap[i]
            seam += int(((got["start"] % cap) + got["length"] > cap).sum())
    assert seam > 0                                                # some asserted window straddles the ring's seam
    assert LENGTHS[0] > 4 * s.planner.out_cap[0]                   # and stream 0 wraps its ring many times


@pytest.mark.parametrize("kind", ["float32", "int16", "mixed"])
def test_resampled_streams_at_mixed_rates(models, kind):
    m = models["bf16"]
    rng = np.random.default_rng(len(kind))
    rates = [44100, 48000, 8000, 32000]
    secs = [31.7, 10.0, 7.5, 23.3]
    recs = []
    for i, (r, sec) in enumerate(zip(rates, secs)):
        pcm = kind == "int16" or (kind == "mixed" and i % 2 == 0)
        recs.append(_signal(int(sec * r) + 17 * i, rng, pcm))
    s = m.open_stream(len(recs), W, 100001, sample_rate=rates, frame_embeddings=True, piece_seconds=3)
    chunked = [_cut(r, rng, s.planner.piece_in[i]) for i, r in enumerate(recs)]
    if kind == "mixed":                                            # float chunks inside an int16 stream too
        chunked[0] = [_as_float(c) if j % 2 else c for j, c in enumerate(chunked[0])]
        recs[0] = torch.cat([_as_float(c) for c in chunked[0]])
    with torch.no_grad():
        calls = _run(s, chunked, rng)
        _check_calls(calls, len(recs))
        for i, rec in enumerate(recs):
            ref = m.forward_windows(rec, W, 100001, frame_embeddings=True, sample_rate=rates[i])
            _assert_equal(_stream_rows(calls, i), ref, (kind, rates[i]))


@pytest.mark.parametrize("pcm", [False, True])
def test_resample_stream_piece_by_piece_equals_resample_of_the_whole(pcm):
    rate = 44100
    rng = np.random.default_rng(3)
    x = _signal(1_234_567, rng, pcm)
    p = StreamPlanner([rate], window=7360, hop=7360, piece_seconds=0.3)
    taps, width, orig, new = preprocess._cached_taps(rate, 32000, torch.device(DEV))
    tf, pg = preprocess.segment_tiling(orig, new, width)
    ring = torch.full((p.ring_len,), float("nan"), device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    sizes = []
    while sum(sizes) < x.numel():
        sizes.append(min(int(rng.integers(1, 30000)), x.numel() - sum(sizes)))
    stitched = []
    at = 0

    def run(piece, chunk):
        if len(piece.append):
            tab = torch.from_numpy(piece.append).to(DEV)
            src = chunk.to(DEV)
            name = "acx_stream_append_pcm16" if src.dtype == torch.int16 else "acx_stream_append"
            _native.call(name, src.data_ptr(), src.numel(), tab.data_ptr(), 1, ring.data_ptr(), ring.numel(), st)
        for rows in piece.resample.values():
            start, n_tiles = preprocess.segment_tiles(rows[:, 4].tolist(), tf, pg, new)
            tab = torch.cat([torch.from_numpy(rows).flatten(), start]).to(DEV)
            _native.call("acx_resample_stream", ring.data_ptr(), ring.numel(), tab.data_ptr(), 1, tab.data_ptr() + 64,
                         n_tiles, taps.data_ptr(), orig, new, width, ring.data_ptr(), ring.numel(), st)
            j = rows[0, 3] * new + np.arange(rows[0, 4])
            stitched.append(ring[torch.from_numpy(p.out_base[0] + j % p.out_cap[0]).to(DEV)].clone())

    for m_ in sizes:
        for (pl,) in p.split([m_]):
            run(p.step([pl]), x[at:at + pl])
            at += pl
    run(p.step([0], [0]), None)
    got = torch.cat(stitched)
    ref = preprocess.resample(x, rate)[0]
    assert got.numel() == ref.numel() == preprocess.resampled_length(x.numel(), rate)
    assert torch.equal(got, ref)


def test_lifecycle_staggered_closes_none_pushes_and_errors(models):
    m = models["bf16"]
    eng = m._get_engine()
    rng = np.random.default_rng(29)
    recs = [_signal(n, rng) for n in (700001, 400000, 1500000, 123456)]
    s = m.open_stream(4, W, 32000, frame_embeddings=False)
    chunked = [_cut(r, rng, s.planner.piece_in[0]) for r in recs]
    with torch.no_grad():
        calls = [s.push([None] * 4)]                               # nothing new anywhere: zero rows
        assert calls[0]["clipwise_logits"].shape == (0, 527) and calls[0]["recording"].numel() == 0
        calls += _run(s, chunked, rng, close_after={1: len(chunked[1]) - 1, 3: len(chunked[3]) - 1})
        for i, rec in enumerate(recs):
            ref = m.forward_windows(rec, W, 32000)
            _assert_equal(_stream_rows(calls, i), ref, i)
    with pytest.raises(ValueError, match="closed"):
        s.push([torch.zeros(10)] + [None] * 3)
    t = m.open_stream(3, W, 32000, sample_rate=[32000, 44100, 8000])
    t.push([torch.zeros(7359), torch.zeros(10000), torch.zeros(1839)])     # 7359 / 7257 / 7356 samples at 32 kHz
    before = eng.launches
    for bad, msg in (([torch.zeros(10)] * 2, "2 chunks for 3"), (torch.zeros(10), "one chunk for 3"),
                     ([torch.zeros(2, 5), None, None], "1-D"), ([torch.zeros(5, dtype=torch.int32), None, None], "dtype")):
        with pytest.raises(ValueError, match=msg):
            t.push(bad)
    for streams in (None, [0], [1], [2]):
        with pytest.raises(ValueError, match="shortest the model takes"):
            t.close(streams)
    assert eng.launches == before and t.closed == [False] * 3
    assert t.planner.n_in == [7359, 10000, 1839]


def test_device_memory_does_not_grow(models):
    m = models["bf16"]
    rng = np.random.default_rng(31)
    s = m.open_stream(2, W, 32000, sample_rate=[32000, 44100])
    one = [_signal(32000, rng).pin_memory(), _signal(44100, rng).pin_memory()]
    with torch.no_grad():
        for _ in range(60):
            s.push(one)
        torch.cuda.synchronize()
        after_1min = torch.cuda.memory_allocated()
        for _ in range(30 * 60 - 60):
            s.push(one)
        torch.cuda.synchronize()
        after_30min = torch.cuda.memory_allocated()
    assert after_30min == after_1min
    assert s.planner.n_in == [30 * 60 * 32000, 30 * 60 * 44100]


def test_full_windows_share_forward_alls_graph(models):
    m = models["bf16"]
    eng = m._get_engine()
    if not eng.use_graph:
        pytest.skip("graphs disabled (ACX_GRAPH=0)")
    eng._ws.clear()
    g = torch.Generator().manual_seed(23)
    x = (torch.randn(eng.chunk, W, generator=g) * 0.1).clamp_(-1, 1).to(DEV)
    recs = (torch.randn(eng.chunk, W, generator=g) * 0.1).clamp_(-1, 1)
    s = m.open_stream(eng.chunk, W, 32000, frame_embeddings=True)
    with torch.no_grad():
        for _ in range(2):
            m.forward_all(x)                                       # captured on the shape's second use
        ws = eng._ws[(eng.chunk, W)]
        graphs, uses = dict(ws["graphs"]), dict(ws["uses"])
        assert (eng.chunk, W, True, True, True, False) in graphs
        res = s.push(list(recs))                                   # exactly one full window per stream: one chunk
        assert res["length"].tolist() == [W] * eng.chunk
        assert eng._ws[(eng.chunk, W)] is ws and ws["graphs"] == graphs and ws["uses"] == uses   # replayed, nothing new
        ref = m.forward_all(recs.to(DEV))
    for k in ("clipwise_logits", "clipwise_output", "scene_embeddings", "frame_embeddings"):
        assert torch.equal(res[k], ref[k]), k


def test_extreme_table_values_stay_inside_their_regions():
    """pos and f0 near 2^63: the kernels reduce / bound them, so every write lands in its row's region."""
    st = torch.cuda.current_stream().cuda_stream
    big = 2 ** 63 - 1
    ring = torch.full((100,), 7.0, device=DEV)
    src = torch.arange(1, 6, dtype=torch.float32, device=DEV)
    tab = torch.tensor([[0, 5, 10, 20, big, 3]], dtype=torch.int64, device=DEV)
    _native.call("acx_stream_append", src.data_ptr(), 5, tab.data_ptr(), 1, ring.data_ptr(), 100, st)
    want = torch.full((100,), 7.0)
    for i in range(5):
        slot = (big % 20 + i) % 20
        want[10 + slot] = i + 1
        if slot < 3:
            want[30 + slot] = i + 1
    assert torch.equal(ring.cpu(), want)

    taps, width, orig, new = preprocess._cached_taps(44100, 32000, torch.device(DEV))
    tf, pg = preprocess.segment_tiling(orig, new, width)
    ring = torch.full((4000,), 7.0, device=DEV)
    ring[:2000] = torch.rand(2000, device=DEV)
    before = ring.clone()
    n_out = 2 * new
    rows = torch.tensor([[0, 2000, 2000, big, n_out, 3000, 500, 100]], dtype=torch.int64)
    start, n_tiles = preprocess.segment_tiles([n_out], tf, pg, new)
    table = torch.cat([rows.flatten(), start]).to(DEV)
    _native.call("acx_resample_stream", ring.data_ptr(), ring.numel(), table.data_ptr(), 1, table.data_ptr() + 64,
                 n_tiles, taps.data_ptr(), orig, new, width, ring.data_ptr(), ring.numel(), st)
    fbase = (1 << 62) // max(orig, new)
    want = before.cpu()
    for j in range(n_out):                                     # input past in_end reads as zero: the outputs are zero
        slot = (fbase * new + j) % 500
        want[3000 + slot] = 0.0
        if slot < 100:
            want[3500 + slot] = 0.0
    assert torch.equal(ring.cpu(), want)


def test_amplitude_check_reads_the_resampled_samples(models, monkeypatch):
    monkeypatch.setenv("ACX_CHECK_AMPLITUDE", "1")
    m = models["bf16"]
    s = m.open_stream(2, W, 32000, sample_rate=[44100, 32000])
    loud = torch.full((44100,), 300.0)
    with pytest.raises(ValueError, match="amplitude"):
        s.push([loud, torch.zeros(32000)])
    t = m.open_stream(2, W, 32000, sample_rate=[44100, 32000])
    with torch.no_grad():
        t.push([torch.full((44100,), 0.5), torch.full((32000,), 0.5)])
