"""GPU (B200): query by example -- each kernel bit for bit against the numpy reference (ties, NaN, +-0, tile edges, range
tables, k past N, millions of keys), a score block of more than 2^31 elements, chunking, search of forward_windows in
both precisions with separation, a query from extract_clipwise, and that validation failures launch nothing."""
import ctypes
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import audioset_convnext_inf_b200 as acx                         # noqa: E402
from audioset_convnext_inf_b200 import _native, search           # noqa: E402
from audioset_convnext_inf_b200.extract import extract_clipwise  # noqa: E402

DEV = "cuda:0"
W = 320000
NAMES = ("acx_row_norms", "acx_cosine_scores", "acx_search_topk")


def _model(sd, prec):
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval().set_precision(prec)


@pytest.fixture(scope="module")
def models(parity_sd):
    return {prec: _model(parity_sd, prec) for prec in ("fp32", "bf16")}


@pytest.fixture
def launches(monkeypatch):
    """Counts the search entry points called through _native.call."""
    seen = []
    real = _native.call

    def counting(name, *args):
        if name in NAMES:
            seen.append(name)
        return real(name, *args)

    monkeypatch.setattr(_native, "call", counting)
    return seen


def _st():
    return torch.cuda.current_stream().cuda_stream


def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


def _awkward(rng, n, d):
    """Keys with exact duplicates (tied scores), a zero vector (NaN), NaN, +-0 and inf entries, and opposite rows."""
    x = rng.standard_normal((n, d)).astype(np.float32)
    for i in range(0, n - 1, 17):
        x[i + 1] = x[i]
    x[2] = 0.0
    x[3, 0] = np.nan
    x[4] = -0.0
    x[5, d - 1] = np.inf
    x[6] = -x[7]
    if d == 1:                                                   # D = 1: every score is +-1, a sea of ties
        x[8:12] = np.float32(0.0)
    return x


def _norms(x):
    t = torch.from_numpy(x).to(DEV)
    buf = torch.full((x.shape[0] + 2,), 7.0, dtype=torch.float64, device=DEV)
    _native.call("acx_row_norms", t.data_ptr(), x.shape[0], x.shape[1], buf[1].data_ptr(), _st())
    assert buf[0].item() == 7.0 and buf[-1].item() == 7.0
    return t, buf[1:-1]


def _scores(q, k):
    qt, qn = _norms(q)
    kt, kn = _norms(k)
    Q, N = q.shape[0], k.shape[0]
    buf = torch.full((Q * N + 64,), 7.0, device=DEV)
    _native.call("acx_cosine_scores", qt.data_ptr(), qn.data_ptr(), Q, kt.data_ptr(), kn.data_ptr(), N, q.shape[1],
                 buf[32].data_ptr(), _st())
    assert (buf[:32] == 7).all() and (buf[-32:] == 7).all()
    return buf[32:-32].view(Q, N)


def _topk(scores, k, ranges=None):
    Q, N = scores.shape
    out_s = torch.full((Q + 2, k), 7.0, device=DEV)
    out_i = torch.full((Q + 2, k), 7, dtype=torch.int64, device=DEV)
    n = ctypes.c_longlong(0)
    _native.call("acx_search_topk_workspace", Q, N, ctypes.addressof(n))
    ws = torch.empty(n.value, dtype=torch.uint8, device=DEV)
    rt = None if ranges is None else torch.from_numpy(ranges).to(DEV)
    _native.call("acx_search_topk", scores.data_ptr(), Q, N, 0 if rt is None else rt.data_ptr(), k, out_s[1].data_ptr(),
                 out_i[1].data_ptr(), ws.data_ptr(), _st())
    for t in (out_s, out_i):
        assert (t[0] == 7).all() and (t[-1] == 7).all()          # sentinels around the outputs
    return out_s[1:-1].cpu().numpy(), out_i[1:-1].cpu().numpy()


def _clamped_neighbours(ranges, N):
    lo = np.clip(ranges[:, 0], 0, N)
    hi = np.clip(ranges[:, 1], 0, N)
    return [np.arange(a, b) for a, b in zip(lo.tolist(), hi.tolist())]


def _pad(score, index, k):
    """reference_topk's (Q, min(k, N)) result padded to k slots, as the kernel writes them."""
    Q, kp = index.shape
    s = np.full((Q, k), np.float32(np.nan), np.float32)
    i = np.full((Q, k), -1, np.int64)
    s[:, :kp], i[:, :kp] = score, index
    return s, i


@pytest.mark.parametrize("d", [1, 7, 768, 769])
def test_kernels_equal_reference(d):
    rng = np.random.default_rng(d)
    Q, N = 67, 301                                               # no multiple of any tile
    keys = _awkward(rng, N, d)
    queries = np.concatenate([keys[[0, 2, 3, 5, 4]], rng.standard_normal((Q - 5, d)).astype(np.float32)])
    _, qn = _norms(queries)
    _, kn = _norms(keys)
    with np.errstate(all="ignore"):
        want_n = np.zeros(N)
        for i in range(d):
            want_n = want_n + keys[:, i].astype(np.float64) ** 2
    assert np.array_equal(kn.cpu().numpy().view(np.uint64), np.sqrt(want_n).view(np.uint64))
    got = _scores(queries, keys)
    ref = search.reference_scores(queries, keys)
    assert np.array_equal(_bits(got.cpu().numpy()), _bits(ref))
    assert np.isnan(ref).any()
    # the order on scores no product makes (a sum from +0.0 is never -0.0): +-0 ties and NaNs of other bit patterns
    ref[:, 20:30:2] = np.float32(-0.0)
    ref[:, 21:31:2] = np.float32(0.0)
    ref[:, 40:44] = np.array([0xffc00000, 0x7f800001, 0x7fc00000, 0xffffffff], np.uint32).view(np.float32)
    ref[:, 50] = np.float32(np.inf)
    ref[:, 51] = np.float32(-np.inf)
    ref[:5, 100:] = ref[:5, 100:101]                             # long runs of ties
    got = torch.from_numpy(ref).to(DEV)
    big = 2 ** 62
    tables = {"empty": np.stack([np.arange(N), np.arange(N)], 1),             # no neighbours at all
              "random": np.sort(rng.integers(-5, N + 5, size=(N, 2)), axis=1),
              "wild": rng.choice(np.array([-big, -1, 0, 3, N - 1, N, N + 1, big]), size=(N, 2))}
    for k in (1, 5, 1024):
        want = _pad(*search.reference_topk(ref, k), k)
        got_s, got_i = _topk(got, k)
        assert np.array_equal(got_i, want[1]) and np.array_equal(_bits(got_s), _bits(want[0])), k
        for name, table in tables.items():
            nb = _clamped_neighbours(table, N)
            want = _pad(*search.reference_topk(ref, k, nb), k)
            got_s, got_i = _topk(got, k, table.astype(np.int64))
            assert np.array_equal(got_i, want[1]) and np.array_equal(_bits(got_s), _bits(want[0])), (k, name)
            if name == "empty":
                assert (got_i[:, :min(k, N)] >= 0).all()


@pytest.mark.parametrize("k", [1, 1024])
def test_topk_over_millions_of_keys(k):
    """Small integer keys: huge runs of tied scores, so the threshold's ties are taken lowest index first."""
    rng = np.random.default_rng(k)
    N, d = 3_000_017, 7
    keys = rng.integers(-2, 3, size=(N, d)).astype(np.float32)
    queries = rng.integers(-2, 3, size=(3, d)).astype(np.float32)
    queries[2] = keys[N - 1]
    got = _scores(queries, keys)
    ref = search.reference_scores(queries, keys)
    sample = rng.integers(0, N, 100000)
    got_sample = got[:, torch.from_numpy(sample).to(DEV)].cpu().numpy()
    assert np.array_equal(_bits(got_sample), _bits(ref[:, sample]))
    got_s, got_i = _topk(got, k)
    want_s, want_i = search.reference_topk(ref, k)
    assert np.array_equal(got_i, want_i) and np.array_equal(_bits(got_s), _bits(want_s))


def test_cosine_scores_past_2_31_elements():
    rng = np.random.default_rng(9)
    Q, N, d = 70, 31_000_000, 2                                  # 2.17e9 scores
    keys = rng.standard_normal((N, d)).astype(np.float32)
    queries = rng.standard_normal((Q, d)).astype(np.float32)
    got = _scores(queries, keys)
    assert Q * N > 2 ** 31
    qs = np.concatenate([rng.integers(0, Q, 4000), [Q - 1] * 8])
    ns = np.concatenate([rng.integers(0, N, 4000), N - 1 - np.arange(8)])
    vals = got[torch.from_numpy(qs).to(DEV), torch.from_numpy(ns).to(DEV)].cpu().numpy()
    want = np.array([search.reference_scores(queries[q:q + 1], keys[n:n + 1])[0, 0] for q, n in zip(qs, ns)])
    assert np.array_equal(_bits(vals), _bits(want))
    del got
    torch.cuda.empty_cache()


def _signal(n, rng):
    return torch.from_numpy(np.clip(rng.standard_normal(n) * 0.1, -1, 1).astype(np.float32))


def _np(d):
    return {c: v.cpu().numpy() for c, v in d.items()}


@pytest.fixture(scope="module")
def recordings():
    rng = np.random.default_rng(3)
    return [_signal(n, rng) for n in (2_400_017, 1_600_000)]    # 75 s and 50 s: two recordings, tails off the grid


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_search_of_forward_windows_equals_reference(models, recordings, prec, launches):
    m = models[prec]
    with torch.no_grad():
        win = m.forward_windows(recordings, W, 32000)
    emb = win["scene_embeddings"]
    torch.manual_seed(4)
    queries = torch.cat([emb[[3, 50, 70]], emb[[10, 60]] + 0.05 * torch.randn(2, emb.shape[1], device=DEV)])
    rows = tuple(win[c].cpu().numpy() for c in ("recording", "start", "length"))
    keys = emb.cpu().numpy()
    N = keys.shape[0]
    for sep in (0, 160000, 320000, sys.maxsize):                # sys.maxsize: one hit per recording
        for k in (1, 20, 1024):
            launches.clear()
            got = _np(search.search(queries, win, k, separation_samples=sep))
            assert launches == ["acx_row_norms", "acx_row_norms", "acx_cosine_scores", "acx_search_topk"]
            want = search.reference_search(queries.cpu().numpy(), keys, k, rows, sep)
            assert got["index"].shape == (5, min(k, N))
            assert np.array_equal(_bits(got["score"]), _bits(want["score"])), (sep, k)
            for c in ("index", "recording", "start", "length"):
                assert got[c].dtype == np.int64 and np.array_equal(got[c], want[c]), (sep, k, c)
            if sep == sys.maxsize:
                assert ((got["index"] >= 0).sum(axis=1) == min(k, 2)).all()
            if sep:
                for q in range(5):                               # the separation property
                    hit = got["index"][q] >= 0
                    r, s = got["recording"][q][hit], got["start"][q][hit]
                    for a in range(len(r)):
                        same = (r == r[a]) & (np.arange(len(r)) != a)
                        assert (np.abs(s[same] - s[a]) >= sep).all()
                # rows of one recording never suppress rows of another: each recording alone gives the same hits
                if k == 1024:
                    for rec in (0, 1):
                        sel = torch.nonzero(win["recording"] == rec).flatten()
                        sub = {c: win[c][sel] for c in ("scene_embeddings", "recording", "start", "length")}
                        alone = _np(search.search(queries, sub, k, separation_samples=sep))
                        for q in range(5):
                            mine = got["index"][q][(got["index"][q] >= 0) & (got["recording"][q] == rec)]
                            other = alone["index"][q][alone["index"][q] >= 0] + int(sel[0])
                            assert sorted(mine.tolist()) == sorted(other.tolist()), (rec, q)


def test_shrunken_chunk_budget_gives_the_same_results(models, recordings, monkeypatch):
    with torch.no_grad():
        win = models["bf16"].forward_windows(recordings, W, 32000)
    N = win["scene_embeddings"].shape[0]
    emb = win["scene_embeddings"]
    queries = torch.cat([emb * 1.5, emb[:42] - 0.25])            # 150 queries
    whole = search.search(queries, win, 50, separation_samples=96000)
    for qc in (4, 100):                                          # chunks of 4, and of 100 rounded down to one 64-query tile
        monkeypatch.setattr(search, "SCORE_BLOCK_BYTES", qc * N * 8)
        parts = search.search(queries, win, 50, separation_samples=96000)
        for c in whole:
            assert torch.equal(whole[c], parts[c]) if c != "score" else \
                np.array_equal(_bits(whole[c].cpu().numpy()), _bits(parts[c].cpu().numpy())), (qc, c)


def test_query_from_extract_clipwise(models, recordings):
    m = models["fp32"]
    clip = recordings[1][32000 * 12:32000 * 12 + W]              # exactly window 12 of recording 1
    q = extract_clipwise(m, [clip.numpy()], want=("scene_embeddings",))["scene_embeddings"][0]
    with torch.no_grad():
        win = m.forward_windows(recordings, W, 32000)
    hits = search.search(q[None].to(DEV), win, 5, separation_samples=160000)
    assert hits["recording"][0, 0].item() == 1 and hits["start"][0, 0].item() == 32000 * 12
    want = search.reference_search(q[None].numpy(), win["scene_embeddings"].cpu().numpy(), 5,
                                   tuple(win[c].cpu().numpy() for c in ("recording", "start", "length")), 160000)
    assert np.array_equal(hits["index"].cpu().numpy(), want["index"])
    assert np.array_equal(_bits(hits["score"].cpu().numpy()), _bits(want["score"]))


def test_validation_failures_launch_nothing(models, recordings, launches):
    with torch.no_grad():
        win = models["bf16"].forward_windows(recordings[1], W, 32000)
    q = win["scene_embeddings"][:2]
    bad_order = dict(win, start=win["start"].flip(0))
    for args, kw in (((q[:, :10], win, 3), {}), ((q, win, 0), {}), ((q, win["scene_embeddings"], 3),
                                                                         {"separation_samples": 5}),
                     ((q, bad_order, 3), {}), ((q, win["scene_embeddings"].cpu(), 3), {}),
                     ((q.double(), win, 3), {}), ((q, win, 3), {"separation_samples": -1})):
        with pytest.raises(ValueError):
            search.search(*args, **kw)
    assert launches == []
    search.search(q, win, 3, separation_samples=64000)
    assert launches == ["acx_row_norms", "acx_row_norms", "acx_cosine_scores", "acx_search_topk"]
