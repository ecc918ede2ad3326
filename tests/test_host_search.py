"""CPU: the host side of query by example -- the numpy reference against an independent per-pair Python loop and a
sorted() order, neighbour ranges against brute force, the separation property, validation, and the argument checks of
the new entry points."""
import ctypes
import math
import sys

import numpy as np
import pytest
import torch

from audioset_convnext_inf_b200 import _native, search
from audioset_convnext_inf_b200.windows import plan_windows

W = 320000


def _pair_score(q, k):
    """One score by the definition, with Python floats (fp64): the same chain, written independently."""
    d = qq = kk = 0.0
    for a, b in zip(q.tolist(), k.tolist()):
        d += a * b
        qq += a * a
        kk += b * b
    with np.errstate(all="ignore"):
        v = np.float32(np.float64(d) / (np.float64(math.sqrt(qq)) * np.float64(math.sqrt(kk))))
    return np.float32(np.nan) if np.isnan(v) else v


def _sort_key(s, i):
    s = float(s)
    return (1, 0.0, i) if math.isnan(s) else (0, -s, i)


def _awkward(rng, n, d):
    """Rows with duplicates (tied scores), zero vectors, NaN, +-0 and inf entries."""
    x = rng.standard_normal((n, d)).astype(np.float32)
    x[1] = x[0]                                                  # a duplicate key: a tie at every query
    x[2] = 0.0                                                   # zero vector: NaN
    x[3, 0] = np.nan
    x[4] = -0.0
    x[5, d - 1] = np.inf
    x[6] = -x[0]
    x[7] = x[0] * np.float32(2)                                  # the same direction: equal scores (mostly)
    x[9] = x[8]
    return x


@pytest.mark.parametrize("d", [1, 3, 17])
def test_reference_scores_equal_a_per_pair_python_loop(d):
    rng = np.random.default_rng(d)
    keys = _awkward(rng, 12, d)
    queries = np.concatenate([keys[[0, 2, 3, 5]], rng.standard_normal((3, d)).astype(np.float32)])
    got = search.reference_scores(queries, keys)
    assert got.dtype == np.float32 and got.shape == (7, 12)
    want = np.array([[_pair_score(q, k) for k in keys] for q in queries], dtype=np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert np.isnan(got[:, 2]).all() and np.isnan(got[1]).all()  # a zero vector on either side
    assert (got[np.isnan(got)].view(np.uint32) == 0x7fc00000).all()


@pytest.mark.parametrize("k", [1, 5, 12, 50])
def test_reference_topk_equals_sorted_order(k):
    rng = np.random.default_rng(k)
    keys = _awkward(rng, 12, 4)
    queries = np.concatenate([keys[[0, 3, 4]], rng.standard_normal((4, 4)).astype(np.float32)])
    s = search.reference_scores(queries, keys)
    s[5, 10] = np.float32(-0.0)                                  # -0 and +0 tie and go by index
    s[5, 11] = np.float32(0.0)
    score, index = search.reference_topk(s, k)
    assert score.shape == index.shape == (7, min(k, 12))
    for q in range(7):
        want = sorted(range(12), key=lambda i: _sort_key(s[q, i], i))[:k]
        assert index[q].tolist() == want
        assert np.array_equal(score[q].view(np.uint32), s[q, want].view(np.uint32))
    assert index[0, :2].tolist() == [0, 1][:k]                   # the duplicate: a tie, the lower index first


def _brute_ranges(rec, start, sep):
    out = []
    for w in range(len(rec)):
        nb = [j for j in range(len(rec)) if rec[j] == rec[w] and abs(int(start[j]) - int(start[w])) < sep]
        out.append(nb)
    return out


@pytest.mark.parametrize("sep", [1, 32000, 160000, 320001, 10 ** 9, sys.maxsize, 2 ** 63, 2 ** 80])
@pytest.mark.parametrize("hop", [32000, 99999])
def test_neighbour_ranges_equal_brute_force(sep, hop):
    lengths = [W + 7 * 32000 + 12345, W - 5, 3 * W + 1, W + hop + 1]  # tails off the hop grid, a short recording
    plan = plan_windows(lengths, W, hop)
    rec, start = plan.recording.numpy(), plan.start.numpy()
    table = search.neighbour_ranges(rec, start, sep)
    assert table.dtype == np.int64 and table.shape == (len(rec), 2)
    for w, nb in enumerate(_brute_ranges(rec, start, sep)):
        assert list(range(*table[w])) == nb, w
    if sep >= 10 ** 9:                                           # wider than every recording: the whole recording
        for w in range(len(rec)):
            assert list(range(*table[w])) == np.flatnonzero(rec == rec[w]).tolist()


def _independent_local_max(s, rec, start, sep):
    """Eligibility and top k by Python comparisons of sort keys, independent of the reference's arrays."""
    out = []
    for q in range(s.shape[0]):
        ok = [w for w in range(len(rec))
              if all(_sort_key(s[q, w], w) < _sort_key(s[q, j], j) for j in range(len(rec))
                     if j != w and rec[j] == rec[w] and abs(int(start[j]) - int(start[w])) < sep)]
        out.append(sorted(ok, key=lambda i: _sort_key(s[q, i], i)))
    return out


@pytest.mark.parametrize("sep", [0, 96000, 160000, 320000, sys.maxsize])
def test_reference_search_separation(sep):
    rng = np.random.default_rng(sep + 1)
    plan = plan_windows([W + 40 * 32000 + 777, 2 * W + 3], W, 32000)
    rec, start, length = (getattr(plan, c).numpy() for c in ("recording", "start", "length"))
    N = len(rec)
    # a smooth walk through embedding space: neighbouring windows are alike, as overlapping windows are
    keys = np.cumsum(rng.standard_normal((N, 8)), axis=0).astype(np.float32)
    keys[5] = keys[6]                                            # tied neighbours
    queries = keys[[3, 30, N - 2]] + rng.standard_normal((3, 8)).astype(np.float32)
    ref = search.reference_search(queries, keys, 40, (rec, start, length), sep)
    s = search.reference_scores(queries, keys)
    want = _independent_local_max(s, rec, start, sep if sep else 1)
    for q in range(3):
        hits = ref["index"][q][ref["index"][q] >= 0].tolist()
        assert hits == want[q][:40]
        assert (ref["index"][q][len(hits):] == -1).all() and np.isnan(ref["score"][q][len(hits):]).all()
        assert ref["recording"][q][:len(hits)].tolist() == rec[hits].tolist()
        assert ref["start"][q][:len(hits)].tolist() == start[hits].tolist()
        assert ref["length"][q][:len(hits)].tolist() == length[hits].tolist()
        assert (ref["start"][q][len(hits):] == -1).all()
        if sep == sys.maxsize:                                   # one hit per recording: its best row
            assert len(hits) == 2 and sorted(rec[hits].tolist()) == [0, 1]
        if sep:
            assert len(hits) < 40                                # a smooth walk has few local maxima
            for a in hits:                                       # the separation property
                for b in hits:
                    if a != b and rec[a] == rec[b]:
                        assert abs(int(start[a]) - int(start[b])) >= sep
        else:
            assert len(hits) == 40


# ---- validation -----------------------------------------------------------------------------------------------------------
def _windows(n=6, d=8, **over):
    plan = plan_windows([W + (n - 1) * 32000], W, 32000)
    w = {"scene_embeddings": torch.rand(plan.start.numel(), d), "recording": plan.recording, "start": plan.start,
         "length": plan.length}
    w.update(over)
    return w


def test_search_validation():
    q = torch.rand(3, 8)
    k = torch.rand(10, 8)
    w = _windows()
    bad = [((q.double(), k, 5), "queries must be a 2-D float32"), ((q[0], k, 5), "queries must be a 2-D float32"),
           ((q, k.half(), 5), "keys must be"), ((q, k[:, :7], 5), "7 dimensions"),
           ((torch.rand(3, 0), torch.rand(10, 0), 5), "at least one dimension"), ((q, k, 0), "k = 0"),
           ((q, k, 1025), "k = 1025"), ((q, k, 2.0), "k = 2.0"), ((q, k, True), "k = True"),
           ((q, k, 5, -1), "separation_samples = -1"), ((q, k, 5, 1.5), "separation_samples"),
           ((q, k, 5, 32000), "needs the windows dict"), ((q, {"scene_embeddings": k}, 5), "lacks"),
           ((q, dict(w, scene_embeddings=w["scene_embeddings"].double()), 5), "scene_embeddings must be"),
           ((q, _windows(start=w["start"].flip(0)), 5), "start ascending"),
           ((q, _windows(recording=torch.tensor([0, 0, 1, 0, 0, 0])), 5), "recording-major"),
           ((q, _windows(length=w["length"][:-1]), 5), "rows, scene_embeddings"),
           ((q, _windows(start=w["start"].int()), 5), "int64"),
           ((q, _windows(length=w["length"] * 0), 5), "length >= 1")]
    for args, msg in bad:
        with pytest.raises(ValueError, match=msg):
            search.search(*args)
    for args in ((q, k, 5), (q, w, 5, 64000), (q, w, 5, sys.maxsize), (q, w, 5, 2 ** 63)):   # every host check passes,
        # then it needs the GPU (any separation is valid: one wider than a recording makes it one neighbourhood)
        with pytest.raises(ValueError, match="CUDA"):
            search.search(*args)


def test_search_refuses_more_than_2_31_keys():
    huge = torch.empty(1, 8).expand(2 ** 31, 8)                  # a view of one row: no memory behind it
    assert huge.shape[0] == 2 ** 31
    with pytest.raises(ValueError, match="at most 2147483647"):
        search.search(torch.rand(1, 8), huge, 5)


# ---- C ABI --------------------------------------------------------------------------------------------------------------
_P = 4096


def test_row_norms_entry_point_rejects_bad_arguments():
    fn = _native.load().acx_row_norms
    assert len(_native.SIGNATURES["acx_row_norms"]) == 5
    for args in ((0, 10, 8, _P, 0), (_P, 10, 8, 0, 0)):
        assert fn(*args) == _native.ACX_ERR_ARG and "row_norms: null" in _native.last_error()
    for args, msg in (((_P, 0, 8, _P, 0), "rows=0"), ((_P, -3, 8, _P, 0), "rows=-3"), ((_P, 10, 0, _P, 0), "d=0"),
                      ((_P, 2 ** 41, 8, _P, 0), "rows=2199023255552")):
        assert fn(*args) == _native.ACX_ERR_ARG and msg in _native.last_error(), args


def _scores_args(q=_P, qn=_P, Q=4, k=_P, kn=_P, N=10, d=8, out=_P):
    return (q, qn, Q, k, kn, N, d, out, 0)


def test_cosine_scores_entry_point_rejects_bad_arguments():
    fn = _native.load().acx_cosine_scores
    assert len(_native.SIGNATURES["acx_cosine_scores"]) == len(_scores_args())
    for kw in (dict(q=0), dict(qn=0), dict(k=0), dict(kn=0), dict(out=0)):
        assert fn(*_scores_args(**kw)) == _native.ACX_ERR_ARG and "cosine_scores: null" in _native.last_error(), kw
    for kw, msg in ((dict(Q=0), "Q=0"), (dict(Q=-1), "Q=-1"), (dict(Q=65535 * 64 + 1), "Q=4194241"),
                    (dict(N=0), "N=0"), (dict(N=-2), "N=-2"), (dict(N=2 ** 31), "N=2147483648"), (dict(d=0), "d=0"),
                    (dict(d=-4), "d=-4")):
        assert fn(*_scores_args(**kw)) == _native.ACX_ERR_ARG and msg in _native.last_error(), kw
    assert fn(*([0] * len(_scores_args()))) == _native.ACX_ERR_ARG


def _topk_args(s=_P, Q=4, N=10, ranges=_P, k=5, out_s=_P, out_i=_P, ws=_P):
    return (s, Q, N, ranges, k, out_s, out_i, ws, 0)


def test_search_topk_entry_points_reject_bad_arguments():
    lib = _native.load()
    fn = lib.acx_search_topk
    assert len(_native.SIGNATURES["acx_search_topk"]) == len(_topk_args())
    for kw in (dict(s=0), dict(out_s=0), dict(out_i=0), dict(ws=0), dict(s=0, ranges=0)):
        assert fn(*_topk_args(**kw)) == _native.ACX_ERR_ARG and "search_topk: null" in _native.last_error(), kw
    for kw, msg in ((dict(Q=0), "Q=0"), (dict(Q=-1), "Q=-1"), (dict(N=0), "N=0"), (dict(N=2 ** 31), "N=2147483648"),
                    (dict(k=0), "k=0"), (dict(k=1025), "k=1025"), (dict(k=-1, ranges=0), "k=-1")):
        assert fn(*_topk_args(**kw)) == _native.ACX_ERR_ARG and msg in _native.last_error(), kw
    assert fn(*([0] * len(_topk_args()))) == _native.ACX_ERR_ARG
    n = ctypes.c_longlong(-1)
    ws = lib.acx_search_topk_workspace
    assert ws(7, 1000, ctypes.addressof(n)) == 0 and n.value == 7 * 1000 * 4
    assert ws(7, 1000, 0) == _native.ACX_ERR_ARG and "null" in _native.last_error()
    for args, msg in (((0, 10), "Q=0"), ((3, 0), "N=0"), ((3, 2 ** 31), "N=2147483648"), ((-1, 5), "Q=-1")):
        assert ws(*args, ctypes.addressof(n)) == _native.ACX_ERR_ARG and msg in _native.last_error(), args
