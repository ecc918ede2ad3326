"""GPU (B200): resampling at any sample rate -- acx_resample_segments, preprocess.resample, and the sample_rate argument
of ConvNeXt.forward_windows and extract.extract_clipwise.

Every segment of a packed buffer must equal acx_resample_fit of that segment alone, BIT FOR BIT, without reading or
writing a sample outside itself; and tagging at any rate must equal tagging the resampled audio at 32 kHz, bit for bit."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import audioset_convnext_inf_b200 as acx                      # noqa: E402
from audioset_convnext_inf_b200 import _native                # noqa: E402
from audioset_convnext_inf_b200.preprocess import (_cached_taps, resample, resample_fit, resampled_length,  # noqa: E402
                                                   segment_tiles, segment_tiling)

DEV = "cuda:0"
W = 320000
KEYS = ("clipwise_logits", "clipwise_output", "scene_embeddings", "frame_embeddings", "frame_lengths", "recording",
        "start", "length")
RATES = (44100, 22050, 48000, 96000, 16000, 8000)
# mixed lengths, several shorter than the filter's width (9 to 41 input samples at these rates)
SEG_LENGTHS = (1, 2, 5, 17, 40, 441, 4410, 32001, 123457, 3, 250000)


def _reference(x, rate):
    """acx_resample_fit of one segment alone, at torchaudio's length (int16: the prep kernels' x / 32767, a true division:
    on the device a Python-scalar divisor would become a reciprocal multiply, so the divisor is a tensor)."""
    xf = torch.div(x.float(), torch.tensor(32767.0, device=x.device)) if x.dtype == torch.int16 else x
    return resample_fit(xf[None].to(DEV), rate, 32000, n_out=None)[0]


def _launch(x, segs, out, rate):
    """acx_resample_segments(_pcm16) over (in_off, in_len, out_off, out_len) rows."""
    taps, width, orig, new = _cached_taps(rate, 32000, x.device)
    frames, groups = segment_tiling(orig, new, width)
    start, n_tiles = segment_tiles([s[3] for s in segs], frames, groups, new)
    table = torch.cat([torch.tensor(segs, dtype=torch.int64).flatten(), start]).to(DEV)
    name = "acx_resample_segments_pcm16" if x.dtype == torch.int16 else "acx_resample_segments"
    _native.call(name, x.data_ptr(), x.numel(), table.data_ptr(), len(segs), table.data_ptr() + 32 * len(segs), n_tiles,
                 taps.data_ptr(), orig, new, width, out.data_ptr(), out.numel(), torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("dtype", [torch.float32, torch.int16])
@pytest.mark.parametrize("rate", RATES)
def test_segments_bit_identical_to_resample_fit_alone(rate, dtype):
    """Segments packed with poison between them (NaN, or full-scale int16) and sentinels around their outputs."""
    g = torch.Generator().manual_seed(rate + (dtype == torch.int16))
    if dtype == torch.int16:
        segs_in = [torch.randint(-20000, 20000, (n,), generator=g, dtype=torch.int16) for n in SEG_LENGTHS]
        poison = 32767
    else:
        segs_in = [torch.randn(n, generator=g) * 0.3 for n in SEG_LENGTHS]
        poison = float("nan")
    gap, sentinel = 97, -12345.0
    parts, outs, rows = [], 0, []
    pos = gap
    parts.append(torch.full((gap,), poison, dtype=dtype))
    for x in segs_in:
        n_out = resampled_length(x.numel(), rate)
        rows.append([pos, x.numel(), outs + gap, n_out])
        parts += [x, torch.full((gap,), poison, dtype=dtype)]
        pos += x.numel() + gap
        outs += gap + n_out
    xbuf = torch.cat(parts).to(DEV)
    out = torch.full((outs + gap,), sentinel, device=DEV)
    _launch(xbuf, rows, out, rate)
    torch.cuda.synchronize()
    keep = torch.ones(out.numel(), dtype=torch.bool, device=DEV)
    for x, (_, _, o, n) in zip(segs_in, rows):
        got = out[o:o + n]
        ref = _reference(x, rate)
        assert got.shape == ref.shape and torch.equal(got, ref), (rate, x.numel())
        assert not torch.isnan(got).any()
        keep[o:o + n] = False
    assert (out[keep] == sentinel).all()                     # nothing written outside the segments


def test_resample_api_mixed_list():
    """Mixed rates, dtypes and devices in one call: views of one buffer, exact lengths, each equal to resample_fit alone;
    a waveform already at 32 kHz is copied unchanged."""
    g = torch.Generator().manual_seed(3)
    f = [torch.randn(n, generator=g) * 0.2 for n in (90569, 7, 300001, 50000)]
    pcm = torch.randint(-9000, 9000, (123457,), generator=g, dtype=torch.int16)
    waves = [f[0], pcm, f[1].to(DEV), f[2].double(), f[3], pcm.to(DEV)]
    rates = [44100, 48000, 22050, 44100, 32000, 32000]
    outs = resample(waves, rates)
    assert [o.numel() for o in outs] == [resampled_length(w.numel(), r) for w, r in zip(waves, rates)]
    assert outs[0].numel() == 65720
    base = outs[0].untyped_storage().data_ptr()
    assert all(o.untyped_storage().data_ptr() == base and o.dtype == torch.float32 and o.is_cuda for o in outs)
    for w, r, o in zip(waves[:4], rates[:4], outs[:4]):
        wf = w if w.dtype == torch.int16 else w.float()
        assert torch.equal(o, _reference(wf.cpu(), r)), r
    assert torch.equal(outs[4], f[3].to(DEV))
    assert torch.equal(outs[5], torch.div(pcm.float(), 32767.0).to(DEV))
    # a single contiguous device buffer is read in place, and one rate for all works
    one = resample(f[2].to(DEV), 44100)
    assert len(one) == 1 and torch.equal(one[0], _reference(f[2], 44100))
    assert resample([], 44100) == []


@pytest.mark.parametrize("rate", RATES)
def test_matches_torchaudio_on_the_cpu(rate):
    """The tolerance of test_resample_fit_matches_torchaudio_then_pad_crop on the common prefix; the exact length."""
    TAF = pytest.importorskip("torchaudio.functional")
    g = torch.Generator().manual_seed(rate)
    waves = [torch.randn(int(rate * s) + 3, generator=g) * 0.3 for s in (0.73, 1.9, 3.0)]
    outs = resample(waves, rate)
    for w, o in zip(waves, outs):
        ref = TAF.resample(w[None], rate, 32000)[0]
        n = min(ref.numel(), o.numel())
        assert o.numel() == resampled_length(w.numel(), rate) and o.numel() - ref.numel() in (0, 1)
        got = o[:n].cpu()
        assert (got - ref[:n]).abs().max().item() < 2e-6 * max(1.0, ref.abs().max().item()) * 5


def test_past_2_31_samples():
    """An int16 48 kHz recording of 3.3e9 samples (6.6 GB; 2.2e9 outputs, 8.8 GB): interior output slices past input
    sample 2^31 and past output sample 2^31 equal resample_fit of an input slice starting at a multiple of orig (3)."""
    n = 3_300_000_000
    g = torch.Generator(device=DEV).manual_seed(29)
    rec = torch.randint(-20000, 20000, (n,), dtype=torch.int16, device=DEV, generator=g)
    out = resample(rec, 48000)[0]
    assert out.numel() == resampled_length(n, 48000) == 2_200_000_000
    checked = 0
    for in_start in (3 * ((2 ** 31 + 123456) // 3), 3 * ((3 * 2 ** 30 + 777) // 3), 3 * ((n - 40000) // 3)):
        sl = rec[in_start:in_start + 30000]
        ref = _reference(sl, 48000)
        j0 = in_start // 3 * 2                               # output index of the slice's first frame
        lo, hi = 40, ref.numel() - 40                        # interior: the K = 23 inputs lie inside the slice
        assert torch.equal(out[j0 + lo:j0 + hi], ref[lo:hi]), in_start
        checked += j0 + lo >= 2 ** 31
    assert checked >= 2
    del rec, out


def _model(sd, prec):
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval().set_precision(prec)


@pytest.fixture(scope="module")
def models(parity_sd):
    return {prec: _model(parity_sd, prec) for prec in ("fp32", "bf16")}


def _mixed_recordings(seed=41):
    g = torch.Generator().manual_seed(seed)
    f441 = (torch.randn(2_000_003, generator=g) * 0.1).clamp_(-1, 1)            # 45 s at 44.1 kHz, float
    pcm48 = torch.randint(-6000, 6000, (1_500_001,), generator=g, dtype=torch.int16)   # 31 s at 48 kHz, int16
    f32k = (torch.randn(400_000, generator=g) * 0.1).clamp_(-1, 1)               # already at 32 kHz
    short = (torch.randn(200_000, generator=g) * 0.1).clamp_(-1, 1)              # 4.5 s at 44.1 kHz: one own-length window
    return [f441, pcm48, f32k, short], [44100, 48000, 32000, 44100]


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_forward_windows_at_any_rate_equals_the_resampled_recordings(models, prec):
    m = models[prec]
    recs, rates = _mixed_recordings()
    resampled = [o.clone() for o in resample(recs, rates)]
    with torch.no_grad():
        got = m.forward_windows(recs, W, 100001, frame_embeddings=True, sample_rate=rates)
        ref = m.forward_windows(resampled, W, 100001, frame_embeddings=True)
    lengths = [resampled_length(r.numel(), sr) for r, sr in zip(recs, rates)]
    assert (got["length"] < W).sum().item() == 1 and got["length"].max().item() == W
    last = got["recording"] == 0
    assert got["start"][last].max().item() + W == lengths[0]                  # planned on the resampled length
    for k in KEYS:
        assert torch.equal(got[k], ref[k]), k


def test_default_rate_launches_no_resampler_and_keeps_int16(models, monkeypatch):
    m = models["bf16"]
    eng = m._get_engine()
    names, bufs = [], []
    real_call, real_run = _native.call, eng.run_windows
    monkeypatch.setattr(_native, "call", lambda name, *a: (names.append(name), real_call(name, *a))[1])
    monkeypatch.setattr(eng, "run_windows", lambda buf, *a: (bufs.append(buf), real_run(buf, *a))[1])
    pcm = torch.randint(-6000, 6000, (700_001,), generator=torch.Generator().manual_seed(5), dtype=torch.int16)
    with torch.no_grad():
        a = m.forward_windows(pcm, W, 100001)
        b = m.forward_windows(pcm, W, 100001, sample_rate=32000)
        c = m.forward_windows([pcm], W, 100001, sample_rate=[32000])
    assert names and not [n for n in names if "resample" in n]
    assert [x.dtype for x in bufs] == [torch.int16] * 3
    for k in ("clipwise_logits", "scene_embeddings", "start"):
        assert torch.equal(a[k], b[k]) and torch.equal(a[k], c[k]), k


def test_validation_failures_launch_nothing(models, monkeypatch):
    m = models["bf16"]
    eng = m._get_engine()
    names = []
    monkeypatch.setattr(_native, "call", lambda name, *a: names.append(name))
    before = eng.launches
    recs, rates = _mixed_recordings()
    too_short = torch.zeros(10_000)                                             # 7257 samples at 32 kHz
    assert resampled_length(10_000, 44100) == 7257
    with pytest.raises(ValueError, match="recording 4 has 7257"):
        m.forward_windows(recs + [too_short], sample_rate=rates + [44100])
    for bad in (rates[:3], 44100.0, 0, [44100, 48000, 32000, "44100"]):
        with pytest.raises(ValueError, match="sample_rate"):
            m.forward_windows(recs, sample_rate=bad)
    with pytest.raises(ValueError, match="shared memory"):
        m.forward_windows(recs, sample_rate=44056)
    with pytest.raises(ValueError, match="clip 1 has 7257"):
        acx.extract.extract_clipwise(m, [recs[0].numpy(), too_short.numpy()], sample_rate=44100)
    with pytest.raises(ValueError, match="shared memory"):
        resample(recs, 44056)
    assert names == [] and eng.launches == before


def test_extract_clipwise_at_44100_equals_the_resampled_clips(models):
    m = models["bf16"]
    rng = np.random.default_rng(19)
    clips = [(rng.standard_normal(int(44100 * s)) * 0.1).astype(np.float32) for s in (0.5, 12.3, 3.0, 25.1, 7.7, 3.0)]
    clips.append(rng.integers(-6000, 6000, size=44100 * 2).astype(np.int16))
    resampled = [o.cpu().numpy() for o in resample([torch.from_numpy(c) for c in clips], 44100)]
    want = ("clipwise_logits", "scene_embeddings", "frame_embeddings", "frame_lengths")
    got = acx.extract.extract_clipwise(m, clips, max_batch=3, want=want, sample_rate=44100)
    ref = acx.extract.extract_clipwise(m, resampled, max_batch=3, want=want)
    for k in want:
        assert len(got[k]) == len(clips)
        for i in range(len(clips)):
            assert torch.equal(got[k][i], ref[k][i]), (k, i)
