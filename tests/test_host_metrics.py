"""CPU: the host side of the tagging metrics -- the vectorised numpy reference against an independent per-group Python
loop, the exact rationals and sklearn; the final divisions and their warning; d'; validation; and the argument checks
of the new entry points."""
import ctypes
import subprocess
import sys
import warnings
from fractions import Fraction

import numpy as np
import pytest
import torch

from audioset_convnext_inf_b200 import _native, metrics

F32_MAX = float(np.finfo(np.float32).max)
DENORMALS = [1e-45, 3e-45, -1e-45, 1.1754942e-38, -1.1754942e-38]


def _per_group(s, y):
    """(P, U2, S, exact AP numerator sum_g p_g TP_g / C_g, G) of one column by a loop over tie groups.  Python floats
    compare -0.0 == 0.0, so the two zeros are one dict key and one group, independently of the reference's bit keys."""
    groups = {}
    for v, t in zip(np.asarray(s, dtype=np.float32).tolist(), np.asarray(y).tolist()):
        g = groups.setdefault(v, [0, 0])
        g[0 if t else 1] += 1
    TP = C = U2 = S = 0
    exact = Fraction(0)
    for v in sorted(groups, reverse=True):
        p, n = groups[v]
        PA = TP
        TP += p
        C += p + n
        U2 += n * (2 * PA + p)
        if p:
            S += (p * TP << 64) // C
            exact += Fraction(p * TP, C)
    return TP, U2, S, exact, len(groups)


def _awkward(rng, n):
    """Columns of n rows: quantised scores (heavy ties), +-0, denormals, +-FLT_MAX, a constant column, a column without
    positives, one without negatives, and an ordinary one."""
    cols, labels = [], []
    q = (np.round(rng.standard_normal(n) * 3) / 3).astype(np.float32)
    cols.append(q)
    labels.append(rng.random(n) < 0.3)
    z = rng.choice(np.array([0.0, -0.0, 1e-45, -1e-45, 0.5], dtype=np.float32), n)
    cols.append(z)
    labels.append(rng.random(n) < 0.5)
    e = rng.choice(np.array([F32_MAX, -F32_MAX, 0.0, *DENORMALS], dtype=np.float32), n)
    cols.append(e)
    labels.append(rng.random(n) < 0.4)
    cols.append(np.full(n, 0.25, dtype=np.float32))
    labels.append(rng.random(n) < 0.5)
    cols.append(rng.random(n).astype(np.float32))
    labels.append(np.zeros(n, dtype=bool))
    cols.append(rng.random(n).astype(np.float32))
    labels.append(np.ones(n, dtype=bool))
    cols.append(rng.standard_normal(n).astype(np.float32))
    labels.append(rng.random(n) < 0.05)
    return np.stack(cols, 1), np.stack(labels, 1).astype(np.uint8)


def _unpack(row):
    P, U2, lo, hi = (int(v) for v in row)
    return P, U2, (hi << 64) | lo


@pytest.mark.parametrize("n", [1, 2, 3, 17, 400, 5000])
def test_reference_counts_equal_per_group_loop(n):
    rng = np.random.default_rng(n)
    s, y = _awkward(rng, n)
    counts = metrics.reference_counts(s, y)
    assert counts.dtype == np.uint64 and counts.shape == (s.shape[1], 4)
    for c in range(s.shape[1]):
        P, U2, S, _, _ = _per_group(s[:, c], y[:, c])
        assert _unpack(counts[c]) == (P, U2, S), c


def test_order_keys():
    s = np.array([-np.inf, -F32_MAX, -1.0, -1e-45, -0.0, 0.0, 1e-45, 1.0, F32_MAX, np.inf], dtype=np.float32)
    k = metrics.order_keys(s)
    assert k.dtype == np.uint32
    assert k[4] == k[5] == 0x80000000                            # -0 is +0
    assert (np.diff(k.astype(np.int64))[[0, 1, 2, 3, 5, 6, 7, 8]] > 0).all()


@pytest.mark.parametrize("seed", range(4))
def test_definitions_equal_exact_rationals(seed):
    rng = np.random.default_rng(100 + seed)
    s, y = _awkward(rng, 300)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        got = metrics.reference_metrics(s, y)
    for c in range(s.shape[1]):
        P, U2, S, exact, G = _per_group(s[:, c], y[:, c])
        Nn = len(s) - P
        assert got["positives"][c] == P
        if P and Nn:
            assert got["auc"][c] == float(Fraction(U2, 2 * P * Nn))
        else:
            assert np.isnan(got["auc"][c])
        if P:
            ap = Fraction(S, P << 64)
            assert got["average_precision"][c] == float(ap)
            assert 0 <= exact / P - ap <= Fraction(G, P << 64)    # the floors' cost
        else:
            assert got["average_precision"][c] == 0.0


def test_reference_matches_sklearn():
    sk = pytest.importorskip("sklearn.metrics")
    rng = np.random.default_rng(7)
    N, K = 3000, 40
    s = (np.round(rng.random((N, K)) * 1000) / 1000).astype(np.float32)          # ties
    s[:, :5] = (np.round(rng.standard_normal((N, 5)) * 2) / 2).astype(np.float32)  # heavy ties, +-0
    s[rng.random((N, K)) < 0.02] *= np.float32(-0.0)
    y = (rng.random((N, K)) < np.linspace(0.002, 0.5, K)).astype(np.uint8)
    y[0] = 1
    y[1] = 0
    got = metrics.reference_metrics(s, y)
    ap = sk.average_precision_score(y, s, average=None)
    auc = sk.roc_auc_score(y, s, average=None)
    assert np.abs(got["average_precision"] - ap).max() < 1e-12
    assert np.abs(got["auc"] - auc).max() < 1e-12
    for c in range(3):                                            # single columns with few rows, the binary code path
        sub = slice(0, 5 + 3 * c)
        yy = y[sub, c].copy()
        yy[:2] = (1, 0)
        one = metrics.reference_metrics(s[sub, c:c + 1], yy[:, None])
        assert abs(one["average_precision"][0] - sk.average_precision_score(yy, s[sub, c])) < 1e-12
        assert abs(one["auc"][0] - sk.roc_auc_score(yy, s[sub, c])) < 1e-12


def test_degenerate_classes_warn_once():
    s = np.random.default_rng(3).random((6, 4)).astype(np.float32)
    y = np.array([[0, 1, 1, 0]] * 6, dtype=np.uint8)
    y[0, 3] = 1
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        got = metrics.reference_metrics(s, y)
    assert len(w) == 1 and w[0].category is RuntimeWarning and "classes [0, 1, 2]" in str(w[0].message)
    assert got["average_precision"][0] == 0.0 and np.isnan(got["auc"][:3]).all()
    assert got["average_precision"][1] == got["average_precision"][2] == 1.0
    assert got["positives"].tolist() == [0, 6, 6, 1] and got["positives"].dtype == np.int64
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        metrics.reference_metrics(s[:, 3:], y[:, 3:])             # no degenerate class: no warning


def test_metrics_from_counts_divides_correctly():
    S = (1 << 94) + 12345
    P, N = 3, 10
    got = metrics.metrics_from_counts(np.array([[P, 41, S & ((1 << 64) - 1), S >> 64]], dtype=np.uint64), N)
    assert got["average_precision"][0] == float(Fraction(S, P << 64))
    assert got["auc"][0] == float(Fraction(41, 2 * P * (N - P)))


def test_d_prime():
    from scipy import stats
    auc = np.array([0.5, 0.973, 0.1, 1.0, 0.0, np.nan])
    d = metrics.d_prime(auc)
    assert d.dtype == np.float64 and d[0] == 0.0 and abs(d[1] - 2.725) < 1e-3
    assert np.array_equal(d[:3], np.sqrt(2.0) * stats.norm.ppf(auc[:3]))
    assert d[3] == np.inf and d[4] == -np.inf and np.isnan(d[5])


def test_package_does_not_import_sklearn():
    code = ("import sys; import audioset_convnext_inf_b200, audioset_convnext_inf.pytorch.evaluate; "
            "from audioset_convnext_inf_b200 import metrics; metrics.reference_counts([[0.5]], [[1]]); "
            "assert 'sklearn' not in sys.modules, 'sklearn imported'")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                       cwd=__import__("os").path.dirname(__import__("os").path.dirname(__file__)))
    assert r.returncode == 0, r.stderr


def test_evaluator_alias():
    from audioset_convnext_inf.pytorch.evaluate import Evaluator
    from audioset_convnext_inf_b200.evalloop import Evaluator as E
    assert Evaluator is E


# ---- validation -----------------------------------------------------------------------------------------------------------
def test_tagging_metrics_validation():
    s = torch.rand(5, 3)
    y = np.zeros((5, 3), dtype=np.uint8)
    bad = [((s.double(), y), "scores must be a 2-D float32"), ((s[0], y), "scores must be a 2-D float32"),
           ((s.numpy(), y), "scores must be a 2-D float32"), ((torch.rand(0, 3), y[:0]), "at least one clip"),
           ((torch.rand(5, 0), y[:, :0]), "at least one clip"), ((s, y[:4]), r"targets of shape \(4, 3\)"),
           ((s, y.T), r"targets of shape \(3, 5\)"), ((s, y.astype(np.float16)), "dtype float16"),
           ((s, torch.zeros(5, 3, dtype=torch.float16)), "dtype torch.float16"),
           ((s, y.astype(np.complex64)), "dtype complex64"), ((s, y.astype(str)), "targets of dtype"),
           ((s, y.astype(object)), "targets of dtype")]
    for args, msg in bad:
        with pytest.raises(ValueError, match=msg):
            metrics.tagging_metrics(*args)
    for t in (y, y.astype(bool), y.astype(np.int64), y.astype(np.uint32), y.astype(np.float64),
              torch.from_numpy(y).float(), torch.from_numpy(y).bool()):
        with pytest.raises(ValueError, match="CUDA"):            # every host check passes; then it needs the GPU
            metrics.tagging_metrics(s, t)


def test_tagging_metrics_refuses_more_than_2_31_clips():
    huge = torch.empty(1, 2).expand(2 ** 31, 2)                  # a view of one row: no memory behind it
    with pytest.raises(ValueError, match="at most 2147483647"):
        metrics.tagging_metrics(huge, huge)


# ---- C ABI --------------------------------------------------------------------------------------------------------------
_P = 4096


def _args(s=_P, N=10, K=7, c0=0, kc=7, t=_P, ws=_P, out=_P):
    return (s, N, K, c0, kc, t, ws, out, 0)


def test_tagging_metrics_entry_points_reject_bad_arguments():
    lib = _native.load()
    fn = lib.acx_tagging_metrics
    assert len(_native.SIGNATURES["acx_tagging_metrics"]) == len(_args())
    for kw in (dict(s=0), dict(t=0), dict(ws=0), dict(out=0)):
        assert fn(*_args(**kw)) == _native.ACX_ERR_ARG and "tagging_metrics: null" in _native.last_error(), kw
    for kw, msg in ((dict(N=0), "N=0"), (dict(N=-1), "N=-1"), (dict(N=2 ** 31), "N=2147483648"), (dict(K=0), "K=0"),
                    (dict(K=-3), "K=-3"), (dict(c0=-1), "classes [-1"), (dict(c0=7, kc=1), "classes [7, 7 + 1)"),
                    (dict(c0=3, kc=5), "classes [3, 3 + 5) outside [0, 7)"), (dict(kc=0), "classes [0, 0 + 0)"),
                    (dict(kc=-2), "classes [0, 0 + -2)"), (dict(kc=8), "classes [0, 0 + 8)")):
        assert fn(*_args(**kw)) == _native.ACX_ERR_ARG and msg in _native.last_error(), kw
    assert fn(*([0] * len(_args()))) == _native.ACX_ERR_ARG
    n = ctypes.c_longlong(-1)
    ws = lib.acx_tagging_metrics_workspace
    assert ws(1000, 7, ctypes.addressof(n)) == 0 and n.value == 7 * (16 * 1000 + 4096)
    assert ws(2 ** 31 - 1, 527, ctypes.addressof(n)) == 0 and n.value == 527 * (16 * (2 ** 31 - 1) + 4096)
    assert ws(1000, 7, 0) == _native.ACX_ERR_ARG and "tagging_metrics_workspace: null" in _native.last_error()
    for args, msg in (((0, 5), "N=0"), ((2 ** 31, 5), "N=2147483648"), ((10, 0), "kc=0"), ((-1, 5), "N=-1")):
        assert ws(*args, ctypes.addressof(n)) == _native.ACX_ERR_ARG and msg in _native.last_error(), args
