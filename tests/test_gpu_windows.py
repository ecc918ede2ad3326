"""GPU (B200): sliding-window tagging of long recordings -- ConvNeXt.forward_windows.

Every window is read in place from the recordings' buffer at its own 64-bit offset, and its outputs must equal a forward
of that window copied out and run alone, BIT FOR BIT, without the window ever reading a sample outside itself."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import audioset_convnext_inf_b200 as acx                      # noqa: E402
from audioset_convnext_inf_b200.engine import out_time_dims   # noqa: E402
from audioset_convnext_inf_b200.windows import plan_windows   # noqa: E402

DEV = "cuda:0"
W = 320000
KEYS = ("clipwise_logits", "clipwise_output", "scene_embeddings")
# 95.3 s (end-aligned tail), exactly 10 s, 7.5 s (one window at its own length), 30 s + 17 samples
LENGTHS = (3049600, W, 240000, 960017)


def _model(sd, prec):
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval().set_precision(prec)


@pytest.fixture(scope="module")
def models(parity_sd):
    return {prec: _model(parity_sd, prec) for prec in ("fp32", "bf16")}


def _recordings(lengths=LENGTHS, seed=5):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(n, generator=g) * 0.1).clamp_(-1, 1) for n in lengths]


def _reference(m, recs, res):
    """forward_all of every window copied out of its recording: full windows stacked into batches, own-length windows
    alone (both equal a run of the window alone)."""
    rec, start, length = (res[k].tolist() for k in ("recording", "start", "length"))
    full = [i for i, n in enumerate(length) if n == W]
    ref = {}
    with torch.no_grad():
        if full:
            x = torch.stack([recs[rec[i]][start[i]:start[i] + W] for i in full]).to(DEV)
            out = m.forward_all(x)
            for j, i in enumerate(full):
                ref[i] = {k: v[j:j + 1] for k, v in out.items()}
        for i, n in enumerate(length):
            if n != W:
                ref[i] = m.forward_all(recs[rec[i]][start[i]:start[i] + n][None].to(DEV))
    return ref


def _assert_rows_equal_reference(res, ref, rows=None):
    h3w = out_time_dims(W)[1][3]
    assert res["frame_embeddings"].shape[2:] == (h3w, 7)
    for i in (range(res["length"].numel()) if rows is None else rows):
        n = int(res["length"][i])
        for k in KEYS:
            assert torch.equal(res[k][i], ref[i][k][0]), (k, i, n)
        h3 = out_time_dims(n)[1][3]
        assert res["frame_lengths"][i].item() == h3
        fr = res["frame_embeddings"][i]
        assert torch.equal(fr[:, :h3], ref[i]["frame_embeddings"][0]), ("frame", i, n)
        assert not fr[:, h3:].any(), ("frame tail not zero", i)


def _assert_plan(res, lengths, hop):
    p = plan_windows(lengths, W, hop)
    for k in ("recording", "start", "length"):
        assert res[k].dtype == torch.int64 and res[k].device == torch.device(DEV)
        assert torch.equal(res[k].cpu(), getattr(p, k)), k


@pytest.mark.parametrize("prec, hop", [("bf16", 32000), ("bf16", 100001), ("bf16", 400000), ("fp32", 100001)])
def test_every_window_bit_identical_to_the_window_alone(models, prec, hop):
    m = models[prec]
    recs = _recordings()
    with torch.no_grad():
        res = m.forward_windows(recs, window_samples=W, hop_samples=hop, frame_embeddings=True)
    _assert_plan(res, LENGTHS, hop)
    assert res["clipwise_logits"].shape == (res["length"].numel(), 527)
    assert res["scene_embeddings"].shape == (res["length"].numel(), 768)
    _assert_rows_equal_reference(res, _reference(m, recs, res))


def test_a_window_never_reads_outside_itself(models):
    """NaN in the gaps a hop > window leaves, and whole NaN recordings next to every other one: nothing changes."""
    m = models["bf16"]
    hop = 400000
    short, long_, tail = _recordings((240000, 3049600, 960017), seed=7)
    nan_rec = torch.full((50000,), float("nan"))
    gappy = long_.clone()
    covered = torch.zeros(gappy.numel(), dtype=torch.bool)
    p = plan_windows([gappy.numel()], W, hop)
    for s in p.start.tolist():
        covered[s:s + W] = True
    assert not covered.all()
    gappy[~covered] = float("nan")
    with torch.no_grad():
        clean = m.forward_windows([short, long_, tail], W, hop, frame_embeddings=True)
        dirty = m.forward_windows([short, nan_rec, gappy, nan_rec, tail], W, hop, frame_embeddings=True)
    keep = [i for i, r in enumerate(dirty["recording"].tolist()) if r in (0, 2, 4)]
    assert len(keep) == clean["length"].numel()
    for k in KEYS + ("frame_embeddings", "frame_lengths", "start", "length"):
        assert torch.equal(dirty[k][keep], clean[k]), k


def test_int16_windows_equal_the_float_path(models):
    m = models["bf16"]
    rng = np.random.default_rng(11)
    lengths = (960017, 200000)                       # one with an end-aligned tail, one short window at its own length
    pcm = [rng.integers(-6000, 6000, size=n).astype(np.int16) for n in lengths]
    flt = [torch.from_numpy((p / 32767.0).astype(np.float32)) for p in pcm]
    with torch.no_grad():
        a = m.forward_windows([torch.from_numpy(p) for p in pcm], W, 100001, frame_embeddings=True)
        b = m.forward_windows(flt, W, 100001, frame_embeddings=True)
        # a device-resident int16 recording is read in place; a mix with a float recording goes through float32
        c = m.forward_windows(torch.from_numpy(pcm[0]).to(DEV), W, 100001, frame_embeddings=True)
        d = m.forward_windows([torch.from_numpy(pcm[0]), flt[1]], W, 100001, frame_embeddings=True)
    assert (a["length"] < W).sum().item() == 1
    for k in KEYS + ("frame_embeddings", "frame_lengths", "recording", "start", "length"):
        assert torch.equal(a[k], b[k]), k
        assert torch.equal(a[k], d[k]), k
        rows = a["recording"] == 0
        assert torch.equal(a[k][rows], c[k]), k


@pytest.mark.parametrize("env", [{"ACX_FRONTEND": "folded"}, {"ACX_FRONTEND": "simt"}])
def test_front_end_routes(parity_sd, monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    m = _model(parity_sd, "bf16")
    assert m._get_engine().frontend == env["ACX_FRONTEND"]
    recs = _recordings((960017, 240000), seed=13)
    rng = np.random.default_rng(13)
    pcm = rng.integers(-6000, 6000, size=700001).astype(np.int16)
    pcm_short = rng.integers(-6000, 6000, size=150001).astype(np.int16)
    with torch.no_grad():
        res = m.forward_windows(recs, W, 100001, frame_embeddings=True)
        res16 = m.forward_windows([torch.from_numpy(pcm), torch.from_numpy(pcm_short)], W, 100001, frame_embeddings=True)
        ref16 = m.forward_windows([torch.from_numpy((p / 32767.0).astype(np.float32)) for p in (pcm, pcm_short)], W, 100001,
                                  frame_embeddings=True)
    _assert_rows_equal_reference(res, _reference(m, recs, res))
    for k in KEYS + ("frame_embeddings",):
        assert torch.equal(res16[k], ref16[k]), k


def test_64_bit_offsets(models):
    """An int16 recording of 2^31 + 10^6 samples (4.3 GB, made on the device): windows past sample 2^31 equal their slices."""
    m = models["bf16"]
    n = 2 ** 31 + 10 ** 6
    g = torch.Generator(device=DEV).manual_seed(17)
    rec = torch.randint(-6000, 6000, (n,), dtype=torch.int16, device=DEV, generator=g)
    hop = 2 ** 29
    with torch.no_grad():
        res = m.forward_windows(rec, W, hop, frame_embeddings=True)
    start = res["start"].tolist()
    assert start == [0, hop, 2 * hop, 3 * hop, 4 * hop, n - W]
    assert sum(s >= 2 ** 31 for s in start) == 2
    x = torch.stack([torch.from_numpy(rec[s:s + W].cpu().numpy().astype(np.float32) / np.float32(32767.0)) for s in start])
    del rec
    with torch.no_grad():
        ref = m.forward_all(x.to(DEV))
    for k in KEYS + ("frame_embeddings",):
        assert torch.equal(res[k], ref[k]), k


def test_full_windows_share_forward_alls_graph(models):
    m = models["bf16"]
    eng = m._get_engine()
    if not eng.use_graph:
        pytest.skip("graphs disabled (ACX_GRAPH=0)")
    hop = 32000
    eng._ws.clear()
    g = torch.Generator().manual_seed(23)
    x = (torch.randn(eng.chunk, W, generator=g) * 0.1).clamp_(-1, 1).to(DEV)
    rec = (torch.randn(W + (eng.chunk - 1) * hop, generator=g) * 0.1).clamp_(-1, 1).to(DEV)   # exactly one chunk of windows
    with torch.no_grad():
        for _ in range(2):
            m.forward_all(x)                            # captured on the shape's second use
        ws = eng._ws[(eng.chunk, W)]
        graphs = dict(ws["graphs"])
        uses = dict(ws["uses"])
        assert (eng.chunk, W, True, True, True, False) in graphs
        res = m.forward_windows(rec, W, hop, frame_embeddings=True)
        assert res["length"].numel() == eng.chunk
        assert eng._ws[(eng.chunk, W)] is ws and ws["graphs"] == graphs and ws["uses"] == uses   # replayed, nothing new
        steps = []
        for _ in range(3):
            m.forward_windows(rec, W, hop)
            steps.append(dict(ws["graphs"]))
    new = (eng.chunk, W, True, True, False, False)
    assert new not in steps[0] and steps[1].keys() == graphs.keys() | {new}
    assert steps[2] == steps[1]
    ref = m.forward_all(torch.stack([rec[s:s + W] for s in res["start"].tolist()]))
    for k in KEYS + ("frame_embeddings",):
        assert torch.equal(res[k], ref[k]), k


def test_bad_arguments_raise_before_any_launch(models):
    m = models["bf16"]
    eng = m._get_engine()
    rec = torch.zeros(400000, device=DEV)
    before = eng.launches
    for kw in (dict(window_samples=7359), dict(hop_samples=0), dict(hop_samples=-1)):
        with pytest.raises(ValueError):
            m.forward_windows(rec, **kw)
    with pytest.raises(ValueError, match="recording 1"):
        m.forward_windows([rec, torch.zeros(7359)])
    with pytest.raises(ValueError, match="1-D"):
        m.forward_windows([rec, torch.zeros(2, 9000)])
    with pytest.raises(ValueError, match="dtype"):
        m.forward_windows(torch.zeros(400000, dtype=torch.int32))
    with pytest.raises(ValueError):
        eng.run_windows(rec, plan_windows([400001], W, 32000), ("logits",))        # plan overruns the buffer
    m.train()
    try:
        with pytest.raises(RuntimeError, match="eval"):
            m.forward_windows(rec)
    finally:
        m.eval()
    assert eng.launches == before
