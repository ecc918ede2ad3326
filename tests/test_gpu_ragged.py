"""GPU (B200): ragged batches -- clips of different lengths in one forward, each computed at its own length.

A clip's result in a ragged batch must equal the clip run alone at its exact length BIT FOR BIT: every kernel that reads
across time rows bounds the clip by its own length, and the sums of valid rows have the same terms in the same order."""
import math
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import audioset_convnext_inf_b200 as acx                      # noqa: E402
from audioset_convnext_inf_b200.engine import MIN_RAGGED_LEN, out_time_dims    # noqa: E402
from oracle import weights                                    # noqa: E402

DEV = "cuda:0"
KEYS = ("clipwise_logits", "clipwise_output", "scene_embeddings")
# the golden tolerances of test_gpu_model.py (parity weights)
TOL = {"fp32": dict(logits=1e-4 * 5, scene=5e-4, frame=2e-3), "bf16": dict(logits=2e-2 * 3, scene=0.12, frame=0.6)}


def _model(sd, prec):
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval().set_precision(prec)


@pytest.fixture(scope="module")
def models(parity_sd):
    return {prec: _model(parity_sd, prec) for prec in ("fp32", "bf16")}


def _lengths_covering_every_case(canvas=352000):
    """The shortest legal clip, the canvas itself, a 10 s clip, and lengths until T hits every residue mod 4 and h0, h1,
    h2 both parities."""
    out = [MIN_RAGGED_LEN, canvas, 320000]
    need = {("T", r) for r in range(4)} | {(f"h{s}", p) for s in range(3) for p in range(2)}

    def cases(n):
        T, hs = out_time_dims(n)
        return {("T", T % 4)} | {(f"h{s}", hs[s] % 2) for s in range(3)}

    for n in out:
        need -= cases(n)
    n = 20000
    while need:
        n += 977                                     # not a multiple of the hop: sample offsets inside a frame vary too
        if cases(n) & need:
            out.append(n)
            need -= cases(n)
    return out


def _canvas(clips, L, fill=0.0):
    x = torch.full((len(clips), L), fill, dtype=torch.float32)
    for b, c in enumerate(clips):
        x[b, :c.numel()] = c
    return x.to(DEV)


def _alone(m, clip):
    with torch.no_grad():
        return m.forward_all(clip[None].to(DEV))


def _assert_clip_equal(res, b, one, n):
    for k in KEYS:
        assert torch.equal(res[k][b], one[k][0]), (k, b, n)
    h3 = out_time_dims(n)[1][3]
    assert res["frame_lengths"][b].item() == h3
    fr = res["frame_embeddings"][b]
    assert torch.equal(fr[:, :h3], one["frame_embeddings"][0]), ("frame", b, n)
    assert not fr[:, h3:].any(), ("frame tail not zero", b, n)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_ragged_batch_bit_identical_to_each_clip_alone_and_never_reads_the_tail(models, prec):
    m = models[prec]
    lengths = _lengths_covering_every_case()
    L = max(lengths)
    g = torch.Generator().manual_seed(5)
    clips = [(torch.randn(n, generator=g) * 0.1).clamp_(-1, 1) for n in lengths]
    with torch.no_grad():
        res = m.forward_all(_canvas(clips, L), lengths=lengths)
        nan = m.forward_all(_canvas(clips, L, float("nan")), lengths=torch.tensor(lengths))
    assert res["frame_embeddings"].shape == (len(lengths), 768, out_time_dims(L)[1][3], 7)
    assert res["frame_lengths"].dtype == torch.int64
    for b, (c, n) in enumerate(zip(clips, lengths)):
        _assert_clip_equal(res, b, _alone(m, c), n)
    for k in KEYS + ("frame_embeddings", "frame_lengths"):       # samples past a clip's end are never read
        assert torch.equal(nan[k], res[k]), k


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_ragged_batch_against_reference_goldens(models, golden_dir, prec):
    demo = np.load(os.path.join(golden_dir, "demo_clip.npz"))
    short = np.load(os.path.join(golden_dir, "synth_short.npz"))
    noise = np.load(os.path.join(golden_dir, "synth_noise.npz"))
    clips = [torch.from_numpy(demo["pcm"].astype(np.float32) / 32768.0),
             weights.make_waveforms(1, n_samples=int(short["n_samples"]), kind="noise", seed=3)[0],
             *weights.make_waveforms(2, kind="noise", seed=0)]
    lengths = [c.numel() for c in clips]
    with torch.no_grad():
        res = {k: v.cpu() for k, v in models[prec].forward_all(_canvas(clips, max(lengths)), lengths=lengths).items()}
    t = TOL[prec]

    def close(got, ref, lim):
        assert got.shape == ref.shape
        assert (got - torch.from_numpy(ref)).abs().max().item() < lim

    close(res["clipwise_logits"][0:1], demo["logits"], t["logits"])
    close(res["clipwise_output"][0:1], demo["probs"], t["logits"])
    close(res["scene_embeddings"][0:1], demo["scene"], t["scene"])
    close(res["frame_embeddings"][0:1], demo["frame"], t["frame"])
    h3 = int(res["frame_lengths"][1])
    close(res["clipwise_logits"][1:2], short["logits"], t["logits"])
    close(res["frame_embeddings"][1:2, :, :h3], short["frame"], t["frame"])
    close(res["clipwise_logits"][2:4], noise["logits"], t["logits"])
    close(res["scene_embeddings"][2:4], noise["scene"], t["scene"])
    close(res["frame_embeddings"][2:4, :, ::int(noise["frame_stride"])], noise["frame_t0"], t["frame"])


@pytest.mark.parametrize("env", [{"ACX_DWCONV": "simt"}, {"ACX_GP": "0"}, {"ACX_LN": "smem"}, {"ACX_DWCONV_TC_STAGES": "0"},
                                 {"ACX_DS_GP": "0"}, {"ACX_DS_FUSED": "0"}, {"ACX_DS_FUSED_C": "96,192,384"}, {"ACX_PDL": "0"},
                                 {"ACX_PDL": "31"}, {"ACX_FRONTEND": "folded"}])
def test_ragged_equals_exact_length_on_every_route(parity_sd, monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    m = _model(parity_sd, "bf16")
    lengths = [MIN_RAGGED_LEN + 333, 41017, 64000, 52311]
    clips = weights.make_waveforms(4, n_samples=64000, kind="tones", seed=3)
    clips = [clips[b, :n] for b, n in enumerate(lengths)]
    with torch.no_grad():
        res = m.forward_all(_canvas(clips, 64000), lengths=lengths)
    for b, (c, n) in enumerate(zip(clips, lengths)):
        _assert_clip_equal(res, b, _alone(m, c), n)


def test_one_graph_serves_every_length_mix_across_chunks(models):
    """More clips than a chunk; three calls on the same canvas with different length mixes: the ragged graphs are
    captured once (second call) and replayed (third), and every result equals the exact-length runs."""
    m = models["bf16"]
    eng = m._get_engine()
    if not eng.use_graph:
        pytest.skip("graphs disabled (ACX_GRAPH=0)")
    L = 48000
    B = eng.chunk + 6
    pool = [MIN_RAGGED_LEN, 12345, 20000, 33333, 40961, L]
    rng = np.random.default_rng(3)
    g = torch.Generator().manual_seed(9)
    eng._ws.clear()
    graphs, runs = [], []
    for call in range(3):                             # the exact-length runs come after: they would evict the workspace
        lengths = rng.choice(pool, size=B).tolist()
        clips = [(torch.randn(n, generator=g) * 0.1).clamp_(-1, 1) for n in lengths]
        with torch.no_grad():
            runs.append((lengths, clips, m.forward_all(_canvas(clips, L), lengths=lengths)))
        graphs.append({k: v[0] for k, v in eng._ws[(eng.chunk, L)]["graphs"].items() if k[-1]})
    assert not graphs[0]                              # first use of the shape runs eagerly
    assert sorted(k[0] for k in graphs[1]) == [6, eng.chunk]
    assert graphs[2].keys() == graphs[1].keys() and all(graphs[2][k] is graphs[1][k] for k in graphs[1])
    assert len({tuple(r[0]) for r in runs}) == 3
    for lengths, clips, res in runs:
        for n in set(lengths):                        # exact-length reference: all clips of one length in one batch
            idx = [b for b, x in enumerate(lengths) if x == n]
            with torch.no_grad():
                ref = m.forward_all(torch.stack([clips[b] for b in idx]).to(DEV))
            for j, b in enumerate(idx):
                _assert_clip_equal(res, b, {k: v[j:j + 1] for k, v in ref.items()}, n)


def test_bad_lengths_raise_before_any_launch(models):
    m = models["bf16"]
    eng = m._get_engine()
    x = torch.zeros(2, 32000, device=DEV)
    before = eng.launches
    for bad in ([7359, 9000], [9000, 32001], [9000]):
        with pytest.raises(ValueError):
            m.forward_all(x, lengths=bad)
    with pytest.raises(ValueError):
        eng.run(x, want=("logmel",), lengths=[9000, 9000])
    assert eng.launches == before


def test_extract_clipwise_batches_ragged_and_equals_the_per_clip_loop(models):
    m = models["bf16"]
    g = torch.Generator().manual_seed(21)
    lengths = [MIN_RAGGED_LEN + 1731 * i for i in range(40)]
    order = torch.randperm(40, generator=g).tolist()
    waves = [(torch.randn(lengths[i], generator=g) * 0.1).numpy() for i in order]
    calls = []
    real = m.forward_all

    def counted(*a, **k):
        calls.append(k.get("lengths"))
        return real(*a, **k)

    m.forward_all = counted
    try:
        res = acx.extract.extract_clipwise(m, waves, max_batch=16,
                                           want=("clipwise_logits", "scene_embeddings", "frame_embeddings"))
    finally:
        del m.forward_all
    assert len(calls) <= math.ceil(40 / 16)
    for i, w in enumerate(waves):
        one = _alone(m, torch.from_numpy(w))
        assert torch.equal(res["clipwise_logits"][i], one["clipwise_logits"][0].cpu())
        assert torch.equal(res["scene_embeddings"][i], one["scene_embeddings"][0].cpu())
        assert torch.equal(res["frame_embeddings"][i], one["frame_embeddings"][0].cpu())
