"""GPU (B200): tagging metrics -- the device counts (P, U2, S) bit for bit against the numpy reference (ties, +-0,
denormals, +-FLT_MAX, constant columns, P = 0 and P = N, every digit pass or none skipped, a score matrix of more than
2^31 elements), invariance under row permutations and class chunking, validation that launches nothing, and the
Evaluator drop-in against sklearn."""
import ctypes
import warnings

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import audioset_convnext_inf_b200 as acx                         # noqa: E402
from audioset_convnext_inf_b200 import _native, evalloop, metrics  # noqa: E402
from oracle import weights                                       # noqa: E402

DEV = "cuda:0"
F32_MAX = float(np.finfo(np.float32).max)


def _st():
    return torch.cuda.current_stream().cuda_stream


def _counts(s, y, kc=None):
    """acx_tagging_metrics over all classes in chunks of kc, out between sentinel rows: (K, 4) uint64."""
    N, K = s.shape
    kc = kc or K
    n = ctypes.c_longlong(0)
    _native.call("acx_tagging_metrics_workspace", N, kc, ctypes.addressof(n))
    ws = torch.empty(n.value, dtype=torch.uint8, device=DEV)
    out = torch.full((K + 2, 4), 7, dtype=torch.int64, device=DEV)
    for c0 in range(0, K, kc):
        _native.call("acx_tagging_metrics", s.data_ptr(), N, K, c0, min(kc, K - c0), y.data_ptr(), ws.data_ptr(),
                     out[1 + c0].data_ptr(), _st())
    out = out.cpu().numpy()
    assert (out[0] == 7).all() and (out[-1] == 7).all()
    return out[1:-1].view(np.uint64)


def _columns(rng, N, K):
    """K columns: sigmoid scores, and for K >= 7 also quantised scores (heavy ties), +-0 / denormals, +-FLT_MAX, a
    constant column, no positives, only positives."""
    s = (1 / (1 + np.exp(-(rng.standard_normal((N, K)) * 3 - 2)))).astype(np.float32)
    y = rng.random((N, K)) < rng.uniform(0.001, 0.5, K)
    if K >= 7:
        s[:, 1] = np.round(rng.standard_normal(N) * 4) / 4
        s[:, 2] = rng.choice(np.array([0.0, -0.0, 1e-45, -1e-45, 1.1754942e-38, 0.75], np.float32), N)
        s[:, 3] = rng.choice(np.array([F32_MAX, -F32_MAX, 0.0, -1.0, 1.0], np.float32), N)
        s[:, 4] = 0.125
        y[:, 5] = False
        y[:, 6] = True
    return s, y.astype(np.uint8)


def _check(s, y, **kw):
    got = _counts(torch.from_numpy(s).to(DEV), torch.from_numpy(y).to(DEV), **kw)
    want = metrics.reference_counts(s, y)
    assert np.array_equal(got, want)
    return got


@pytest.mark.parametrize("K", [1, 7, 527])
@pytest.mark.parametrize("N", [1, 2, 255, 4097, 20371])
def test_counts_equal_reference(N, K):
    rng = np.random.default_rng(N * 1000 + K)
    s, y = _columns(rng, N, K)
    _check(s, y)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        got = metrics.tagging_metrics(torch.from_numpy(s).to(DEV), y)
        want = metrics.reference_metrics(s, y)
    for name in ("average_precision", "auc", "positives"):
        assert np.array_equal(got[name].view(np.uint64 if got[name].dtype == np.float64 else np.int64),
                              want[name].view(np.uint64 if want[name].dtype == np.float64 else np.int64)), name


@pytest.mark.parametrize("step", [1 / 1024, 1 / 16, 1.0])
def test_quantised_scores(step):
    """Scores on a grid: few, large tie groups that straddle the 2048-record tiles of the sort and the scan."""
    rng = np.random.default_rng(int(1 / step))
    N, K = 20371, 33
    s = (np.round(rng.random((N, K)) / step) * step).astype(np.float32)
    y = (rng.random((N, K)) < 0.3).astype(np.uint8)
    _check(s, y)


def test_digit_passes_skipped_or_not():
    """Columns where every byte of the key varies (no pass skipped), where only the low bytes vary (the high passes
    skipped), where one byte varies, and where every pass is skipped (a constant column)."""
    rng = np.random.default_rng(5)
    N = 9000
    bits = rng.integers(0, 2 ** 32, N, dtype=np.uint64).astype(np.uint32)
    full = bits.view(np.float32).copy()
    full[~np.isfinite(full)] = 1.0
    low = (np.uint32(0x3f000000) | (bits & np.uint32(0xffff))).view(np.float32)
    mid = (np.uint32(0x3f000000) | (bits & np.uint32(0xff00))).view(np.float32)
    s = np.stack([full, low, mid, np.full(N, -3.5, np.float32), -full], 1)
    y = (rng.random(s.shape) < 0.2).astype(np.uint8)
    _check(s, y)


def test_row_order_and_chunking_do_not_matter(monkeypatch):
    rng = np.random.default_rng(11)
    N, K = 5000, 61
    s, y = _columns(rng, N, K)
    s[:, 10:20] = np.round(s[:, 10:20] * 8) / 8
    base = _check(s, y)
    for seed in range(3):
        perm = np.random.default_rng(seed).permutation(N)
        assert np.array_equal(_counts(torch.from_numpy(s[perm]).to(DEV), torch.from_numpy(y[perm]).to(DEV)), base)
    for kc in (1, 5, 32, 33, 60):
        assert np.array_equal(_counts(torch.from_numpy(s).to(DEV), torch.from_numpy(y).to(DEV), kc), base)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        whole = metrics.tagging_metrics(torch.from_numpy(s).to(DEV), y)
        monkeypatch.setattr(metrics, "METRICS_BLOCK_BYTES", 16 * N * 7)     # chunks of 7 classes
        chunked = metrics.tagging_metrics(torch.from_numpy(s).to(DEV), y)
    for name in whole:
        assert np.array_equal(whole[name], chunked[name], equal_nan=name == "auc")


def test_more_than_2_31_elements():
    """N K > 2^31: the record, row and histogram offsets are 64-bit.  The reference runs on the first and last classes
    (the last reads rows past element 2^31)."""
    N, K = 2 ** 22 + 3, 513
    assert N * K > 2 ** 31
    g = torch.Generator(device=DEV).manual_seed(3)
    s = torch.rand(N, K, generator=g, device=DEV)
    s = torch.round(s * 4096) / 4096
    y = (torch.rand(N, K, generator=g, device=DEV) < 0.1).to(torch.uint8)
    got = metrics.tagging_metrics(s, y)
    cols = [0, 1, 255, K - 2, K - 1]
    want = metrics.reference_metrics(s[:, cols].cpu().numpy(), y[:, cols].cpu().numpy())
    for name in ("average_precision", "auc", "positives"):
        assert np.array_equal(got[name][cols], want[name]), name
    del s, y
    torch.cuda.empty_cache()


def test_target_types_agree():
    rng = np.random.default_rng(2)
    s, y = _columns(rng, 700, 9)
    st = torch.from_numpy(s).to(DEV)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        base = metrics.tagging_metrics(st, y)
    assert len(w) == 1 and "classes [5, 6]" in str(w[0].message)
    for t in (y.astype(bool), y.astype(np.int64), y.astype(np.uint32), y.astype(np.float32), y.astype(np.float64),
              torch.from_numpy(y).to(DEV), torch.from_numpy(y).bool().to(DEV), torch.from_numpy(y).double().to(DEV),
              torch.from_numpy(y.astype(np.int32))):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            got = metrics.tagging_metrics(st, t)
        for name in base:
            assert np.array_equal(got[name], base[name], equal_nan=True), (name, t.dtype)


def test_validation_launches_nothing(monkeypatch):
    seen = []
    real = _native.call

    def counting(name, *args):
        seen.append(name)
        return real(name, *args)

    monkeypatch.setattr(_native, "call", counting)
    s = torch.rand(50, 4, device=DEV)
    y = np.zeros((50, 4), np.uint8)
    y[0] = 1
    bad_scores = []
    for v in (float("nan"), float("inf"), float("-inf")):
        b = s.clone()
        b[17, 2] = v
        bad_scores.append(b)
    for b in bad_scores:
        with pytest.raises(ValueError, match="NaN or infinite"):
            metrics.tagging_metrics(b, y)
    for v, dt in ((2, np.uint8), (-1, np.int64), (0.5, np.float32), (np.nan, np.float64), (3, np.int8)):
        t = y.astype(dt)
        t[9, 1] = v
        with pytest.raises(ValueError, match="other than 0 and 1"):
            metrics.tagging_metrics(s, t)
        with pytest.raises(ValueError, match="other than 0 and 1"):
            metrics.tagging_metrics(s, torch.from_numpy(t).to(DEV))
    with pytest.raises(ValueError, match="other than 0 and 1"):
        metrics.tagging_metrics(s, np.full((50, 4), 2 ** 64 - 1, np.uint64))
    with pytest.raises(ValueError, match="targets of shape"):
        metrics.tagging_metrics(s, torch.zeros(50, 5, device=DEV))
    assert seen == []


def _model(sd):
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval().set_precision("fp32")


def test_evaluator_equals_metrics_of_forward_and_sklearn(parity_sd):
    sk = pytest.importorskip("sklearn.metrics")
    m = _model(parity_sd)
    rng = np.random.default_rng(9)
    B, n_batches = 16, 4
    waves = weights.make_waveforms(B * n_batches, n_samples=32000, kind="noise", seed=21).numpy()
    target = (rng.random((B * n_batches, 527)) < 0.2).astype(np.float32)
    target[0], target[1] = 1, 0                                  # every class has a positive and a negative
    loader = [{"waveform": waves[i:i + B], "target": target[i:i + B]} for i in range(0, B * n_batches, B)]
    stats = evalloop.Evaluator(m).evaluate(loader)
    assert set(stats) == {"average_precision", "auc", "d_prime"}
    out = evalloop.forward(m, loader, return_target=True)
    want = metrics.tagging_metrics(torch.from_numpy(out["clipwise_output"]).to(DEV), out["target"])
    for name in ("average_precision", "auc"):
        assert stats[name].dtype == np.float64 and stats[name].shape == (527,)
        assert np.array_equal(stats[name], want[name]), name
    assert np.array_equal(stats["d_prime"], metrics.d_prime(want["auc"]))
    assert np.abs(stats["average_precision"] - sk.average_precision_score(target, out["clipwise_output"],
                                                                          average=None)).max() < 1e-12
    assert np.abs(stats["auc"] - sk.roc_auc_score(target, out["clipwise_output"], average=None)).max() < 1e-12
    from audioset_convnext_inf.pytorch.evaluate import Evaluator
    with pytest.raises(ValueError, match="no \"target\""):
        Evaluator(m).evaluate([{"waveform": waves[:B]}])
