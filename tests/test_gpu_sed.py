"""GPU (B200): sound event detection -- the two kernels against the numpy reference (exactly, ties at thresholds and NaN
included), 64-bit indexing past 2^31 activity elements, sed.detect of forward_windows in both precisions, and the
stream contract: every stream's activity rows and events from all push / close calls equal sed.detect of the whole
stream, bit for bit."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import audioset_convnext_inf_b200 as acx                         # noqa: E402
from audioset_convnext_inf_b200 import _native, sed             # noqa: E402

DEV = "cuda:0"
W = 320000
C = 527


def _model(sd, prec):
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval().set_precision(prec)


@pytest.fixture(scope="module")
def models(parity_sd):
    return {prec: _model(parity_sd, prec) for prec in ("fp32", "bf16")}


@pytest.fixture
def launches(monkeypatch):
    """Counts the detection entry points called through _native.call."""
    seen = []
    real = _native.call

    def counting(name, *args):
        if name in ("acx_window_activity", "acx_detect_events"):
            seen.append(name)
        return real(name, *args)

    monkeypatch.setattr(_native, "call", counting)
    return seen


def _np(d):
    return {k: v.cpu().numpy() for k, v in d.items()}


def test_window_activity_equals_reference_with_poison_and_sentinels():
    rng = np.random.default_rng(1)
    P = 300
    probs = rng.choice(np.array([0.1, 0.25, 0.5, 0.7, 1.0, 3e-8], np.float32), size=(P, C))
    probs += rng.random((P, C), dtype=np.float32) * np.float32(1e-3)
    rows = []
    for _ in range(2000):                                       # rings inside P, reads that wrap their seam
        cap = int(rng.integers(1, 40))
        base = int(rng.integers(0, P - cap + 1))
        rows.append((int(rng.integers(0, 3 * cap)), int(rng.integers(1, cap + 1)), base, cap))
    table = np.array(rows, np.int64)
    poison = np.full((P, C), np.nan, np.float32)
    want = np.empty((len(rows), C), np.float32)
    for m, (first, n, base, cap) in enumerate(rows):
        idx = [base + (first + t) % cap for t in range(n)]
        poison[idx] = probs[idx]                                 # rows a bin may read; everything else stays NaN
        s = probs[idx[0]].copy()
        for i in idx[1:]:
            s = (s + probs[i]).astype(np.float32)
        want[m] = s / np.float32(n)
    buf = torch.full((len(rows) + 2, C), 7.0, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    src = torch.from_numpy(poison).to(DEV)
    tab = torch.from_numpy(table).to(DEV)
    _native.call("acx_window_activity", src.data_ptr(), P, tab.data_ptr(), len(rows), buf[1].data_ptr(), st)
    got = buf.cpu().numpy()
    assert (got[0] == 7).all() and (got[-1] == 7).all()           # sentinels around the output
    assert np.array_equal(got[1:-1], want)                        # bit for bit (no NaN: every read row is real)
    # extreme table values stay inside probs; a bin with n = 0 is NaN
    big = 2 ** 62
    tab = torch.tensor([[big, big, -big, big], [-5, 0, 3, 4]], dtype=torch.int64, device=DEV)
    out = torch.full((2, C), 7.0, device=DEV)
    _native.call("acx_window_activity", src.data_ptr(), P, tab.data_ptr(), 2, out.data_ptr(), st)
    assert torch.isnan(out[1]).all()


LEVELS = np.array([0.1, 0.3, 0.5, 0.7, np.nan], dtype=np.float32)


def test_detect_events_kernel_equals_carried_state_reference():
    """Three sequences in one launch per call, each fed its bins in its own random splits, then closed; ties at on /
    off, NaN, per-class thresholds, a partial last bin, merges and the duration filter."""
    rng = np.random.default_rng(2)
    R = 1000
    nbs = [90, 1, 37]
    n = [nb * R - 400 for nb in nbs]
    tracks = [LEVELS[rng.integers(0, 5, size=(nb, C))] for nb in nbs]
    for t in tracks:
        t[rng.random(t.shape) < 0.5] = np.float32(0.1)
    on = rng.choice(np.array([0.5, 0.7], np.float32), C)
    off = np.minimum(on, rng.choice(np.array([0.3, 0.5], np.float32), C))
    d = sed.Detection(R, on, off, min_duration_samples=2 * R, merge_gap_samples=2 * R + 1)
    state = sed.new_state(3, DEV)
    ref = [sed.EventTracks(d) for _ in nbs]
    done = [0] * 3
    got_all, want_all = [], []
    for call in range(8):
        close = call == 7
        parts, seq, row0 = [], [], 0
        for s, nb in enumerate(nbs):
            b = nb if close else min(nb - 1, done[s] + int(rng.integers(0, 25)))
            b = max(b, done[s])
            parts.append(tracks[s][done[s]:b])
            limit = n[s] if close else b * R
            seq.append((10 + s, row0, b - done[s], done[s], limit, int(close)))
            want_all += [(10 + s, c, o, f, p) for c, o, f, p in ref[s].step(tracks[s][done[s]:b], done[s], limit, close)]
            row0 += b - done[s]
            done[s] = b
        act = torch.from_numpy(np.concatenate(parts)).to(DEV)
        ev = _np(sed.detect_events(act, np.array(seq, np.int64), d, state))
        got = list(zip(*(ev[k].tolist() for k in sed.EVENT_KEYS)))
        assert [g[:2] for g in got] == sorted(g[:2] for g in got)  # ordered (sequence, class, onset)
        got_all += got
    want_all.sort(key=lambda e: (e[0], e[1], e[2]))
    got_all.sort(key=lambda e: (e[0], e[1], e[2]))
    assert len(got_all) == len(want_all) > 0
    assert [(r, c, o, f, np.float32(p)) for r, c, o, f, p in got_all] == \
           [(r, c, o, f, np.float32(p)) for r, c, o, f, p in want_all]
    assert (state[0][0] == 0).all()                              # every track idle after close


def test_activity_past_2_31_elements():
    M = 4_100_000                                                # 2.16e9 activity elements
    P = 64
    probs = torch.rand(P, C, device=DEV)
    m = torch.arange(M, dtype=torch.int64)
    table = torch.stack([m % P, 1 + m % 3, torch.zeros_like(m), torch.full_like(m, P)], 1).numpy()
    act = sed.window_activity(probs, table)
    assert act.shape == (M, C)
    pn = probs.cpu().numpy()
    for row in (0, 1, 2, M // 2, M - 3, M - 2, M - 1):
        first, count = row % P, 1 + row % 3
        s = pn[first].copy()
        for t in range(1, count):
            s = (s + pn[(first + t) % P]).astype(np.float32)
        assert np.array_equal(act[row].cpu().numpy(), s / np.float32(count)), row
    del act
    torch.cuda.empty_cache()


def _signal(n, rng):
    return torch.from_numpy(np.clip(rng.standard_normal(n) * 0.1, -1, 1).astype(np.float32))


def _detection_for(activity):
    """Per-class thresholds from the activity's own quantiles, so that every track has events to find."""
    a = activity.astype(np.float64)
    on = np.quantile(a, 0.7, axis=0).astype(np.float32)
    off = np.minimum(on, np.quantile(a, 0.5, axis=0).astype(np.float32))
    return on, off


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_detect_of_forward_windows_equals_reference(models, prec, launches):
    m = models[prec]
    rng = np.random.default_rng(3)
    recs = [_signal(n, rng) for n in (3049600, 240000, 960017)]
    with torch.no_grad():
        win = m.forward_windows(recs, W, 32000)
    host = _np({k: win[k] for k in ("clipwise_output", "recording", "start", "length")})
    ref_act = sed.reference_activity(host["clipwise_output"], host["recording"], host["start"], host["length"], 16000)
    on, off = _detection_for(ref_act["activity"])
    d = sed.Detection(16000, on, off, min_duration_samples=32000, merge_gap_samples=48000)
    out = sed.detect(win, d)
    assert launches == ["acx_window_activity", "acx_detect_events", "acx_detect_events"]
    got = _np(out["activity"])
    for k in sed.ACTIVITY_KEYS:
        assert np.array_equal(got[k], ref_act[k]), k
    ref_ev = sed.reference_events(ref_act, d)
    ev = _np(out["events"])
    assert len(ev["onset"]) > 100
    for k in sed.EVENT_KEYS:
        assert ev[k].dtype == ref_ev[k].dtype and np.array_equal(ev[k], ref_ev[k]), k
    assert all(v.device == win["clipwise_output"].device for v in out["activity"].values())
    whole = sed.detect(win, sed.Detection(10 ** 9, 0.5))          # R >= n: the recording-level tags
    tags = whole["activity"]["activity"].cpu().numpy()
    assert tags.shape == (3, C) and whole["activity"]["length"].tolist() == [3049600, 240000, 960017]


def _cut(rec, rng):
    out, at = [], 0
    while at < rec.numel():
        m = (1, 32000, 700000, int(rng.integers(1, 60000)), int(rng.integers(1, 500000)))[int(rng.integers(5))]
        out.append(rec[at:at + m])
        at += m
    return out


@pytest.mark.parametrize("prec, R, hop", [("bf16", 32000, 32000), ("bf16", 45001, 100001), ("fp32", 16000, 32000)])
def test_stream_activity_and_events_equal_detect_of_the_whole_stream(models, prec, R, hop):
    m = models[prec]
    rng = np.random.default_rng(R + hop)
    rates = [32000, 44100, 48000, 32000, 44100]
    secs = [61.3, 40.2, 23.7, 7.5, 30.0]                        # stream 3 is shorter than a window
    recs = [_signal(int(s * r), rng) for s, r in zip(secs, rates)]
    with torch.no_grad():
        probe = m.forward_windows(recs[0], W, hop)
    on, off = _detection_for(probe["clipwise_output"].cpu().numpy())
    d = sed.Detection(R, on, off, min_duration_samples=R, merge_gap_samples=R + 7)
    s = m.open_stream(len(recs), W, hop, sample_rate=rates, piece_seconds=3, detection=d)
    assert torch.isnan(s.row_ring).all() and s.detection_bytes > 0
    chunked = [_cut(r, rng) for r in recs]
    close_after = {4: len(chunked[4]) // 2}                      # closed early: the rest is never pushed
    recs[4] = torch.cat(chunked[4][:close_after[4] + 1])
    calls = []
    with torch.no_grad():
        for t in range(max(len(c) for c in chunked)):
            calls.append(s.push([c[t] if t < len(c) and not s.closed[i] else None for i, c in enumerate(chunked)]))
            if t == close_after[4]:
                calls.append(s.close(4))
        calls.append(s.close())
        for i, rec in enumerate(recs):
            ref = sed.detect(m.forward_windows(rec, W, hop, sample_rate=rates[i]), d)
            a = {k: torch.cat([c["activity"][k][c["activity"]["recording"] == i] for c in calls])
                 for k in sed.ACTIVITY_KEYS}
            for k in ("activity", "start", "length"):
                assert torch.equal(a[k], ref["activity"][k]), (i, k)
            ev = {k: torch.cat([c["events"][k][c["events"]["recording"] == i] for c in calls]) for k in sed.EVENT_KEYS}
            key = ev["class"].cpu().numpy() * 2 ** 40 + ev["onset"].cpu().numpy()
            order = torch.from_numpy(np.argsort(key, kind="stable")).to(DEV)
            assert ev["onset"].numel() == ref["events"]["onset"].numel() > 0, i
            for k in sed.EVENT_KEYS[1:]:
                assert torch.equal(ev[k][order], ref["events"][k]), (i, k)
    for c in calls:                                              # each call: stream-major, then (class, onset)
        r, cl = c["events"]["recording"].tolist(), c["events"]["class"].tolist()
        assert list(zip(r, cl)) == sorted(zip(r, cl))


def test_detection_none_changes_nothing(models, launches):
    m = models["bf16"]
    rng = np.random.default_rng(4)
    x = _signal(15 * 32000, rng)
    eng = m._get_engine()
    s = m.open_stream(1, W, 32000)
    with torch.no_grad():
        n0 = eng.launches
        res = s.push(x)
        n_plain = eng.launches - n0
        res_close = s.close()
    assert set(res) == set(res_close) == {"clipwise_output", "clipwise_logits", "scene_embeddings", "recording", "start",
                                          "length"}
    assert launches == [] and s.detection_bytes == 0
    t = m.open_stream(1, W, 32000, detection=sed.Detection(32000, 0.5))
    with torch.no_grad():
        n0 = eng.launches
        res = t.push(x)
        assert eng.launches - n0 == n_plain
    assert set(res) == {"clipwise_output", "clipwise_logits", "scene_embeddings", "recording", "start", "length",
                        "activity", "events"}
    assert t.detection_bytes == t.bins.cap * C * 4 + C * (3 * 8 + 4)


def test_validation_failures_launch_nothing(models, launches):
    m = models["bf16"]
    rng = np.random.default_rng(5)
    with torch.no_grad():
        win = m.forward_windows(_signal(700000, rng), W, 32000)
        gaps = m.forward_windows(_signal(2_000_000, rng), 100000, 150000)
    d = sed.Detection(32000, 0.5)
    bad = dict(win)
    bad["start"] = win["start"].flip(0)
    for w in (bad, gaps, {k: v for k, v in win.items() if k != "length"}):
        with pytest.raises(ValueError):
            sed.detect(w, d)
    with pytest.raises(ValueError):
        m.open_stream(hop_samples=W + 1, detection=d)
    assert launches == []
    sed.detect(gaps, sed.Detection(10 ** 8, 0.5))                # one bin covers the gaps
    assert launches == ["acx_window_activity", "acx_detect_events", "acx_detect_events"]
