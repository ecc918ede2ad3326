"""Tagging metrics on the GPU: per-class average precision, ROC AUC and d' of clipwise scores against labels, the numbers
the reference's Evaluator computes with sklearn's average_precision_score / roc_auc_score (average=None).

metrics.tagging_metrics(scores, targets) returns per-class "average_precision", "auc" (float64) and "positives"
(int64).  Every quantity is an exact integer until one final division, so the results do not depend on row order,
class chunking, launch shape or GPU, and are bit-identical to the numpy reference below.

Definitions (the numpy reference below is these written out; per class c, s = scores[:, c] fp32 finite, y = targets[:, c]
in {0, 1}, N rows):

  P = sum y, Nn = N - P.
  Order key.  -0.0 is mapped to +0.0; then key = u ^ 0x80000000 if the sign bit of the bit pattern u is clear, else ~u,
  so keys compare as unsigned integers in the order of the scores.  Rows of equal key form a tie group; groups are
  ordered by descending key.  For group g: p_g positives, n_g negatives, TP_g = positives in groups >= g, C_g = rows in
  groups >= g, PA_g = TP_g - p_g.
  AUC.  U2 = sum_g n_g (2 PA_g + p_g) (Mann-Whitney, a tie counted as one half; below 2^61 for N < 2^31) and
  auc = U2 / (2 P Nn), rounded once to fp64; NaN when P = 0 or Nn = 0.
  AP.  S = sum over g with p_g > 0 of floor(p_g TP_g 2^64 / C_g) (below 2^95) and ap = S / (P 2^64), rounded once to
  fp64; 0.0 when P = 0.  Summing floors makes S an integer, so it can be reduced in any order; the floors cost at most
  G 2^-64 / P with G groups (<= 1.2e-10 at N = 2^31).  With q, r = divmod(p TP, C) (p TP < 2^62) the fraction is
  floor(r 2^64 / C) = f1 2^32 + f2, f1 = (r << 32) // C, f2 = (((r << 32) % C) << 32) // C, every step within int64
  because r < C < 2^31; S = (sum q << 64) + (sum f1 << 32) + sum f2.
  d' = sqrt(2) * Phi^-1(auc) per class (scipy.stats.norm.ppf), on the host.

These equal sklearn 1.9's average_precision_score and roc_auc_score to within a few ulps: AP is sklearn's step-wise
precision-recall sum with the ties of a score taken as one threshold, AUC its trapezoidal ROC area.  Like sklearn, a
class without positives gets AP 0.0 and AUC NaN and a class without negatives AUC NaN; one RuntimeWarning lists them.

Device work (acx_tagging_metrics, csrc/metrics.cu), per chunk of kc classes: a pack kernel transposes the chunk's
columns into class-major 64-bit records (key << 32 | label) and counts every byte of every key, then one block per
class radix-sorts its records by descending key (skipping a byte whose histogram has a single non-empty bin) and walks
the tie groups.  Memory: 16 N + 4096 bytes of workspace per class of a chunk, kc = min(K, max(1, METRICS_BLOCK_BYTES //
(16 N))).  The checks of the scores and targets need one device-to-host synchronisation and the (K, 4) counts one copy
back."""
import ctypes
import math
import warnings

import numpy as np
import torch

from . import _native

# Workspace of one chunk of classes (16 N bytes per class).  4 GiB holds all 527 classes up to N = 509 k rows.  At the
# 2 M rows of AudioSet's unbalanced train set it gives chunks of 134 classes, fewer blocks than the B200's 148 SMs: on one
# B200 that took 109 ms against 104 ms for one 17 GB chunk of all 527 classes, and 1 GiB chunks (33 classes) took 402 ms
# (tools/bench_metrics.py, DESIGN.md).
METRICS_BLOCK_BYTES = 4 << 30
MAX_N = 2 ** 31 - 1
_M64 = (1 << 64) - 1
_TARGET_DTYPES = {torch.bool, torch.uint8, torch.int8, torch.int16, torch.int32, torch.int64, torch.float32,
                  torch.float64} | {getattr(torch, n) for n in ("uint16", "uint32", "uint64") if hasattr(torch, n)}


def _scores(scores):
    if not isinstance(scores, torch.Tensor) or scores.dim() != 2 or scores.dtype != torch.float32:
        raise ValueError("scores must be a 2-D float32 tensor (clips, classes)")
    if scores.shape[0] < 1 or scores.shape[1] < 1:
        raise ValueError(f"scores of shape {tuple(scores.shape)}: need at least one clip and one class")
    if scores.shape[0] > MAX_N:
        raise ValueError(f"{scores.shape[0]} clips: at most {MAX_N}")
    return scores


def _targets(targets, shape):
    """targets as a tensor (where it was, or on the host for an array): bool, any int type, float32 or float64."""
    if not isinstance(targets, torch.Tensor):
        arr = np.asarray(targets)
        if arr.dtype.kind not in "biu" and arr.dtype not in (np.float32, np.float64):
            raise ValueError(f"targets of dtype {arr.dtype}: expected bool, an int type, float32 or float64")
        if arr.dtype.kind == "u" and arr.dtype != np.uint8:
            arr = arr.astype(np.int64)               # a value past 2^63 wraps negative and is still rejected below
        targets = torch.from_numpy(np.ascontiguousarray(arr))
    elif targets.dtype not in _TARGET_DTYPES:
        raise ValueError(f"targets of dtype {targets.dtype}: expected bool, an int type, float32 or float64")
    if tuple(targets.shape) != tuple(shape):
        raise ValueError(f"targets of shape {tuple(targets.shape)}, scores of shape {tuple(shape)}")
    return targets


def tagging_metrics(scores, targets):
    """Per-class average precision and ROC AUC; see the module docstring for the definitions.

    scores: (N, K) float32 CUDA tensor, every value finite.  targets: (N, K) tensor or array of bool, an int type,
    float32 or float64, every value 0 or 1 (a CPU one is uploaded).  Returns "average_precision" and "auc" as (K,)
    float64 numpy arrays and "positives" (K,) int64.  Shape, dtype and device are checked before anything runs on the
    GPU, and non-finite scores or targets other than 0 / 1 are found with one synchronisation before any metric kernel
    is launched (ValueError)."""
    scores = _scores(scores)
    targets = _targets(targets, scores.shape)
    if not scores.is_cuda:
        raise ValueError("scores must be on a CUDA device: the metrics run on the GPU")
    if targets.is_cuda and targets.device != scores.device:
        raise ValueError(f"targets are on {targets.device}, scores on {scores.device}")
    targets = targets.to(scores.device)
    if targets.dtype not in (torch.bool, torch.uint8, torch.int8, torch.int16, torch.int32, torch.int64,
                             torch.float32, torch.float64):
        targets = targets.to(torch.int64)             # torch's uint16 / 32 / 64: compared as int64
    if targets.dtype == torch.bool:
        binary = torch.ones((), dtype=torch.bool, device=scores.device)
    elif targets.dtype == torch.uint8:
        binary = (targets <= 1).all()
    else:
        binary = ((targets == 0) | (targets == 1)).all()
    finite_ok, binary_ok = torch.stack([torch.isfinite(scores).all(), binary]).tolist()
    if not finite_ok:
        raise ValueError("scores hold NaN or infinite values")
    if not binary_ok:
        raise ValueError("targets hold values other than 0 and 1")
    N, K = scores.shape
    scores = scores.contiguous()
    targets = targets.to(torch.uint8).contiguous()
    kc = min(K, max(1, METRICS_BLOCK_BYTES // (16 * N)))
    ws = torch.empty(workspace_bytes(N, kc), dtype=torch.uint8, device=scores.device)
    out = torch.empty(K, 4, dtype=torch.int64, device=scores.device)
    st = torch.cuda.current_stream(scores.device).cuda_stream
    for c0 in range(0, K, kc):
        _native.call("acx_tagging_metrics", scores.data_ptr(), N, K, c0, min(kc, K - c0), targets.data_ptr(),
                     ws.data_ptr(), out[c0].data_ptr(), st)
    return metrics_from_counts(out.cpu().numpy().view(np.uint64), N)


def workspace_bytes(N, kc):
    n = ctypes.c_longlong(0)
    _native.call("acx_tagging_metrics_workspace", N, kc, ctypes.addressof(n))
    return n.value


def metrics_from_counts(counts, n_rows):
    """The final divisions: (K, 4) uint64 counts (P, U2, S mod 2^64, S >> 64) of n_rows rows -> the tagging_metrics
    dict.  Python int / int rounds correctly.  Warns once (RuntimeWarning) about classes with P = 0 or Nn = 0."""
    counts = np.asarray(counts, dtype=np.uint64)
    K = counts.shape[0]
    ap, auc = np.empty(K), np.empty(K)
    degenerate = []
    for c, (P, U2, lo, hi) in enumerate(counts.tolist()):
        Nn = n_rows - P
        ap[c] = ((hi << 64) | lo) / (P << 64) if P else 0.0
        auc[c] = U2 / (2 * P * Nn) if P and Nn else math.nan
        if not (P and Nn):
            degenerate.append(c)
    if degenerate:
        warnings.warn(f"{len(degenerate)} classes have no positive or no negative clips; their AUC is NaN (and AP 0.0 "
                      f"without positives): classes {degenerate}", RuntimeWarning, stacklevel=3)
    return {"average_precision": ap, "auc": auc, "positives": counts[:, 0].astype(np.int64)}


def d_prime(auc):
    """d' = sqrt(2) * Phi^-1(auc), elementwise, float64 (NaN stays NaN, AUC 0 / 1 give -inf / inf)."""
    from scipy import stats
    return np.sqrt(2.0) * stats.norm.ppf(np.asarray(auc, dtype=np.float64))


# ---- numpy reference ----------------------------------------------------------------------------------------------------
def order_keys(scores):
    """The order key of every score: uint32 of the same shape."""
    u = np.ascontiguousarray(scores, dtype=np.float32).view(np.uint32)
    u = np.where(u == np.uint32(0x80000000), np.uint32(0), u)
    return np.where(u >> np.uint32(31) != 0, ~u, u | np.uint32(0x80000000))


def reference_counts(scores, targets):
    """The definitions written out, one class at a time, vectorised over its tie groups: (K, 4) uint64 counts
    (P, U2, S mod 2^64, S >> 64), the layout acx_tagging_metrics writes."""
    keys = order_keys(scores)
    y = np.asarray(targets) != 0
    N, K = keys.shape
    out = np.zeros((K, 4), dtype=np.uint64)
    for c in range(K):
        order = np.argsort(keys[:, c], kind="stable")[::-1]            # descending key
        k = keys[order, c]
        tp = np.cumsum(y[order, c], dtype=np.int64)
        end = np.flatnonzero(np.append(k[1:] != k[:-1], True))        # the last row of every group
        TP = tp[end]
        C = end + 1
        PA = np.concatenate([[0], TP[:-1]])
        p = TP - PA
        n = (C - np.concatenate([[0], C[:-1]])) - p
        U2 = int(np.sum(n * (2 * PA + p)))
        m = p > 0
        Cm = C[m]
        q, r = np.divmod(p[m] * TP[m], Cm)
        f1, r2 = np.divmod(r << 32, Cm)
        f2 = (r2 << 32) // Cm
        S = (int(q.sum()) << 64) + (int(f1.sum()) << 32) + int(f2.sum())
        out[c] = (int(tp[-1]), U2, S & _M64, S >> 64)
    return out


def reference_metrics(scores, targets):
    """tagging_metrics written out on the host: metrics_from_counts(reference_counts(scores, targets), N)."""
    return metrics_from_counts(reference_counts(scores, targets), np.asarray(scores).shape[0])
