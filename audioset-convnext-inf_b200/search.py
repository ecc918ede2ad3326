"""Query by example: "where else in these 24 hours does it sound like this?", "which of my clips sound like this one?".

search.search(queries, keys, k, separation_samples=0) ranks the rows of `keys` (scene embeddings: a tensor, or the dict
forward_windows / open_stream returns) by exact cosine similarity to each query and returns the best k per query, with
at most one hit per moment of a recording when a separation is given.  Results are bit-identical to the numpy reference
below, on any GPU and at any shape.

Definitions (the numpy reference below is these written out literally):

  Score.  For a query q and a key row k of D dimensions, d = sum_i q_i k_i, qq = sum_i q_i^2 and kk = sum_i k_i^2, each
  sum taken in fp64 over i = 0 .. D-1 in order, starting from 0.0, and
      score = float32(d / (sqrt(qq) * sqrt(kk))),
  every operation IEEE fp64 with round-to-nearest, the conversion round-to-nearest-even; a NaN score is stored as the
  canonical quiet NaN (0x7fc00000).  The product of two fp32 values is exact in fp64, so the GPU's fma(x, y, acc) equals
  acc + x * y in numpy bit for bit and the whole chain is reproducible, which an fp32 FMA chain (or a cuBLAS product,
  whose rounding depends on the algorithm it picks) is not.  A zero vector gives 0 / 0 = NaN; inf or NaN entries give
  what IEEE gives.

  Order.  Hit a beats hit b when score_a > score_b, or the scores are equal and index_a < index_b.  -0.0 equals +0.0;
  NaN ranks below every number, and NaNs are equal to each other (ties go to the lower index).  This is a strict total
  order, so the top k' = min(k, N) hits are unique.

  Separation (a windows dict and separation_samples > 0; 0 is off).  Two rows are neighbours when they belong to the
  same recording and |start_a - start_b| < separation_samples.  A row is eligible for a query when it beats every one of
  its neighbours.  The results are the top k' eligible rows, so any two hits of one query in one recording start at
  least separation_samples apart.  This is local-maximum selection, not greedy non-maximum suppression: a row beaten by
  a neighbour that is itself beaten by a better neighbour is not eligible, so it may return fewer hits than greedy NMS
  would (unused slots hold index -1 and score NaN).  In exchange every row's eligibility depends on its neighbours only,
  so it is deterministic and needs no sequential pass.

Device work, per call: acx_row_norms once for all queries and once for all keys, then per chunk of Qc queries
acx_cosine_scores into a (Qc, N) fp32 score block and acx_search_topk over it (scores are materialised because a row's
eligibility reads neighbours on both sides, across any tile boundary).  Memory: the score block and a key block of the
same size, 8 Qc N bytes together with Qc = max(1, SCORE_BLOCK_BYTES // (8 N)) (256 MiB; rounded down to whole 64-query
score tiles when it exceeds one), 8 (Q + N) bytes of norms and, with separation, the 16 N-byte neighbour range table.  Output shapes are known on the host, so the work needs no device-to-host
synchronisation."""
import ctypes
import numbers

import numpy as np
import torch

from . import _native
from .windows import check_rows

SCORE_BLOCK_BYTES = 256 << 20       # bytes of one chunk's scratch: (Qc, N) fp32 scores plus (Qc, N) 32-bit keys
MAX_K = 1024
MAX_N = 2 ** 31 - 1
_MAX_QC = 65535 * 64                # queries one acx_cosine_scores launch takes
_TILE_Q = 64                        # queries of one acx_cosine_scores tile
_NAN32 = np.float32(np.nan)


def _int(v, name, low, high=None):
    if isinstance(v, bool) or not isinstance(v, numbers.Integral) or int(v) < low or (high is not None and int(v) > high):
        raise ValueError(f"{name} = {v!r}: expected an int in [{low}, {'inf' if high is None else high}]")
    return int(v)


def _matrix(x, name):
    if not isinstance(x, torch.Tensor) or x.dim() != 2 or x.dtype != torch.float32:
        raise ValueError(f"{name} must be a 2-D float32 tensor")
    if x.shape[1] < 1:
        raise ValueError(f"{name} must have at least one dimension per row")
    return x


# ---- host planning ------------------------------------------------------------------------------------------------------
def neighbour_ranges(rec, start, separation):
    """(N, 2) int64 table (lo, hi): the neighbours of row w are the rows in [lo, hi) other than w -- the rows of its
    recording whose start is within separation - 1 samples of its own.  rec / start are checked rows (recording-major,
    start ascending within a recording), so each neighbourhood is a contiguous run.  separation may be any int >= 0,
    however large (sys.maxsize is "one hit per recording")."""
    rec = np.asarray(rec, dtype=np.int64)
    start = np.asarray(start, dtype=np.int64)
    N = len(rec)
    out = np.empty((N, 2), dtype=np.int64)
    edges = np.flatnonzero(np.diff(rec)) + 1
    for a, b in zip(np.concatenate([[0], edges]).tolist(), np.concatenate([edges, [N]]).tolist()):
        s = start[a:b]
        # any separation beyond the recording's start span makes the whole recording a neighbourhood; clamping it (as a
        # Python int) first keeps s +- sep inside int64 for every separation a caller can pass
        sep = min(int(separation), int(s[-1] - s[0]) + 1)
        out[a:b, 0] = a + np.searchsorted(s, s - sep, side="right")
        out[a:b, 1] = a + np.searchsorted(s, s + sep, side="left")
    return out


# ---- device work --------------------------------------------------------------------------------------------------------
def row_norms(x):
    """acx_row_norms: (R,) float64 norms of the rows of a (R, D) float32 CUDA tensor."""
    out = torch.empty(x.shape[0], dtype=torch.float64, device=x.device)
    if x.shape[0]:
        _native.call("acx_row_norms", x.data_ptr(), x.shape[0], x.shape[1], out.data_ptr(),
                     torch.cuda.current_stream(x.device).cuda_stream)
    return out


def _stage(table, device):
    return torch.from_numpy(np.ascontiguousarray(table, dtype=np.int64)).pin_memory().to(device, non_blocking=True)


def search(queries, keys, k, separation_samples=0):
    """The top k keys of every query by exact cosine similarity; see the module docstring for the definitions.

    queries: (Q, D) float32 CUDA tensor.  keys: a (N, D) float32 tensor on the same device, or the dict forward_windows
    (or an open_stream call) returns, whose "scene_embeddings" are the keys and whose "recording" / "start" / "length"
    come with each hit.  k: an int in [1, 1024]; k' = min(k, N).  separation_samples: an int >= 0, > 0 only with a
    windows dict.

    Returns, on the queries' device, "score" (Q, k') float32 and "index" (Q, k') int64 (the key row), and with a windows
    dict also "recording", "start" and "length" (Q, k') int64 gathered by index.  Column 0 is the best hit; unused slots
    (only with separation) hold index -1, score NaN and -1 in the gathered columns.  Every argument is checked on the host
    before any launch (ValueError, nothing launched).  The work itself needs no device-to-host synchronisation; only the
    row check reads a windows dict's recording / start / length to the host, as sed.detect does."""
    queries = _matrix(queries, "queries")
    windows = None
    if isinstance(keys, dict):
        missing = [c for c in ("scene_embeddings", "recording", "start", "length") if c not in keys]
        if missing:
            raise ValueError(f"windows dict lacks {missing}")
        windows, keys = keys, _matrix(keys["scene_embeddings"], "scene_embeddings")
    else:
        keys = _matrix(keys, "keys")
    if keys.shape[1] != queries.shape[1]:
        raise ValueError(f"keys have {keys.shape[1]} dimensions, queries {queries.shape[1]}")
    k = _int(k, "k", 1, MAX_K)
    sep = _int(separation_samples, "separation_samples", 0)
    if sep and windows is None:
        raise ValueError("separation_samples > 0 needs the windows dict (recording and start of every key)")
    Q, D = queries.shape
    N = keys.shape[0]
    if N > MAX_N:
        raise ValueError(f"{N} keys: at most {MAX_N}")
    if windows is not None:
        rec, start, _ = check_rows(windows, N, "scene_embeddings")
    if not queries.is_cuda:
        raise ValueError("queries must be on a CUDA device: search runs on the GPU")
    if keys.device != queries.device:
        raise ValueError(f"keys are on {keys.device}, queries on {queries.device}")
    dev = queries.device
    kp = min(k, N)
    out = {"score": torch.empty(Q, kp, dtype=torch.float32, device=dev),       # every slot written by acx_search_topk
           "index": torch.empty(Q, kp, dtype=torch.int64, device=dev)}
    if Q and kp:
        queries, keys = queries.contiguous(), keys.contiguous()
        ranges = _stage(neighbour_ranges(rec, start, sep), dev) if sep else None
        st = torch.cuda.current_stream(dev).cuda_stream
        qn, kn = row_norms(queries), row_norms(keys)
        Qc = min(Q, max(1, SCORE_BLOCK_BYTES // (8 * N)), _MAX_QC)
        if Qc < Q and Qc > _TILE_Q:
            Qc -= Qc % _TILE_Q                                   # whole 64-query score tiles in every chunk but the last
        scores = torch.empty(Qc, N, dtype=torch.float32, device=dev)
        ws_bytes = _workspace_bytes(Qc, N)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        for q0 in range(0, Q, Qc):
            qb = min(Qc, Q - q0)
            _native.call("acx_cosine_scores", queries[q0].data_ptr(), qn[q0].data_ptr(), qb, keys.data_ptr(),
                         kn.data_ptr(), N, D, scores.data_ptr(), st)
            _native.call("acx_search_topk", scores.data_ptr(), qb, N, 0 if ranges is None else ranges.data_ptr(), kp,
                         out["score"][q0].data_ptr(), out["index"][q0].data_ptr(), ws.data_ptr(), st)
    if windows is not None:
        hit = out["index"] >= 0
        at = out["index"].clamp(min=0)
        for c in ("recording", "start", "length"):
            out[c] = torch.where(hit, windows[c].to(dev)[at], -1)
    return out


def _workspace_bytes(Q, N):
    n = ctypes.c_longlong(0)
    _native.call("acx_search_topk_workspace", Q, N, ctypes.addressof(n))
    return n.value


# ---- numpy reference ----------------------------------------------------------------------------------------------------
def reference_scores(queries, keys):
    """The score definition written out: (Q, N) float32, every sum a loop over i of fp64 arrays from 0.0."""
    q = np.asarray(queries, dtype=np.float32).astype(np.float64)
    kx = np.asarray(keys, dtype=np.float32).astype(np.float64)
    d = np.zeros((q.shape[0], kx.shape[0]))
    qq = np.zeros(q.shape[0])
    kk = np.zeros(kx.shape[0])
    with np.errstate(all="ignore"):
        for i in range(q.shape[1]):
            d = d + q[:, i, None] * kx[None, :, i]
            qq = qq + q[:, i] * q[:, i]
            kk = kk + kx[:, i] * kx[:, i]
        s = (d / (np.sqrt(qq)[:, None] * np.sqrt(kk)[None, :])).astype(np.float32)
    s[np.isnan(s)] = _NAN32
    return s


def beats(sa, ia, sb, ib):
    """The order, elementwise: hit (sa, ia) beats hit (sb, ib)."""
    na, nb = np.isnan(sa), np.isnan(sb)
    return np.where(na, nb & (ia < ib), nb | (sa > sb) | ((sa == sb) & (ia < ib)))


def reference_topk(scores, k, neighbours=None):
    """The top k' = min(k, N) eligible rows of every row of a (Q, N) float32 score matrix: (score, index) numpy arrays of
    shape (Q, k'), padded with NaN / -1.  neighbours[w] lists the neighbours of row w (None: no separation); a row is
    eligible when it beats every neighbour, compared one by one; eligible rows are ranked by np.lexsort((index, -score))
    (NaN sorts last)."""
    scores = np.asarray(scores, dtype=np.float32)
    Q, N = scores.shape
    kp = min(k, N)
    eligible = np.ones((Q, N), dtype=bool)
    if neighbours is not None:
        for w in range(N):
            nb = np.asarray([j for j in neighbours[w] if j != w], dtype=np.int64)
            if len(nb):
                eligible[:, w] = beats(scores[:, w, None], w, scores[:, nb], nb[None, :]).all(axis=1)
    out_s = np.full((Q, kp), _NAN32, dtype=np.float32)
    out_i = np.full((Q, kp), -1, dtype=np.int64)
    for q in range(Q):
        idx = np.flatnonzero(eligible[q])
        order = idx[np.lexsort((idx, -scores[q, idx]))][:kp]
        out_i[q, :len(order)] = order
        out_s[q, :len(order)] = scores[q, order]
    return out_s, out_i


def reference_search(queries, keys, k, rows=None, separation=0):
    """search() written out: reference_scores, neighbours found by comparing every pair of rows (same recording and
    |start_a - start_b| < separation), reference_topk, and with rows = (recording, start, length) of the keys the
    gathered columns."""
    s = reference_scores(queries, keys)
    neighbours = None
    if separation:
        rec, start = (np.asarray(c) for c in rows[:2])
        neighbours = [np.flatnonzero((rec == rec[w]) & (np.abs(start - start[w]) < separation)) for w in range(len(rec))]
    score, index = reference_topk(s, k, neighbours)
    out = {"score": score, "index": index}
    if rows is not None:
        for name, col in zip(("recording", "start", "length"), rows):
            out[name] = np.where(index >= 0, np.asarray(col)[np.maximum(index, 0)], -1)
    return out
