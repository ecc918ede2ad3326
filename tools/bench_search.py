"""Query by example on the GPU: what search.search and each of its kernels cost, the scoring kernel's fp64 rate next to
torch.mm in float64 of the same shape, and the fp32 normalize + mm + topk shortcut it replaces.

  python tools/bench_search.py [--queries 1,100,1000] [--library 1000000] [--k 20] [--reps 5]

Prints one JSON line with the GPU's name and power limit (read in the same run).  Keys are seeded 768-d embeddings made
like overlapping windows' (a moving sum of 10 noise rows plus a shared mean, so neighbouring rows are alike); queries are
keys plus noise.  Windows are 10 s at a 1 s hop in one recording: 3 600 keys for 1 h, 86 400 for 24 h; separation is 0,
10 s or 1 h (at most one hit per hour: a neighbourhood of 7 199 rows, the whole recording for 1 h).  The library is
--library clips (no separation) with 1 000 queries.

  kernels    CUDA events around --reps launches after a warm-up: acx_row_norms over the keys, acx_cosine_scores over all
             queries at once (its fp64 FLOP/s = 2 Q N D / time), acx_search_topk over that block.  The keys of 24 h
             (265 MB) and the library (3.1 GB) are larger than the 126 MB L2; those of 1 h (11 MB) are not.
  search     search.search end to end (k = --k), median of --reps calls, host clock around the call and a synchronise
  mm_f64     torch.mm in float64 of the scoring shape, CUDA events, same run
  baseline   F.normalize(q) @ F.normalize(k).T + topk in fp32: time (as search), and how many of its top-k indices
             are not in the exact top k (separation 0)"""
import argparse
import json
import os
import statistics
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from audioset_convnext_inf_b200 import search   # noqa: E402
from bench_windows import gpu_info              # noqa: E402

D, W, HOP = 768, 320000, 32000
HOUR = 3600 * 32000


def embeddings(n, seed, device):
    g = torch.Generator(device=device).manual_seed(seed)
    noise = torch.randn(n + 9, D, generator=g, device=device)
    c = torch.cat([torch.zeros(1, D, device=device), noise.cumsum(0)])
    mean = torch.randn(D, generator=g, device=device)
    return ((c[10:] - c[:-10]) / 10 ** 0.5 + 2 * mean).contiguous()


def gpu_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def host_ms(fn, reps):
    fn()
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        times.append(1e3 * (time.perf_counter() - t0))
    return statistics.median(times), out


def kernels(queries, keys, ranges, k, reps):
    Q, N = queries.shape[0], keys.shape[0]
    st = torch.cuda.current_stream().cuda_stream
    qn, kn = search.row_norms(queries), search.row_norms(keys)
    scores = torch.empty(Q, N, device=keys.device)
    ws = torch.empty(search._workspace_bytes(Q, N), dtype=torch.uint8, device=keys.device)
    out_s = torch.empty(Q, k, device=keys.device)
    out_i = torch.empty(Q, k, dtype=torch.int64, device=keys.device)
    t_norm = gpu_ms(lambda: search._native.call("acx_row_norms", keys.data_ptr(), N, D, kn.data_ptr(), st), reps)
    t_score = gpu_ms(lambda: search._native.call("acx_cosine_scores", queries.data_ptr(), qn.data_ptr(), Q,
                                                 keys.data_ptr(), kn.data_ptr(), N, D, scores.data_ptr(), st), reps)
    t_topk = gpu_ms(lambda: search._native.call("acx_search_topk", scores.data_ptr(), Q, N,
                                                0 if ranges is None else ranges.data_ptr(), k, out_s.data_ptr(),
                                                out_i.data_ptr(), ws.data_ptr(), st), reps)
    del scores, ws
    torch.cuda.empty_cache()
    return {"row_norms_ms": round(t_norm, 4), "cosine_scores_ms": round(t_score, 4),
            "cosine_scores_tflops_f64": round(2 * Q * N * D / (t_score * 1e-3) / 1e12, 2),
            "search_topk_ms": round(t_topk, 4)}


def mm_f64(queries, keys, reps):
    q64, k64 = queries.double(), keys.double().t()
    out = torch.empty(queries.shape[0], keys.shape[0], dtype=torch.float64, device=keys.device)
    t = gpu_ms(lambda: torch.mm(q64, k64, out=out), reps)
    res = {"mm_f64_ms": round(t, 4),
           "mm_f64_tflops": round(2 * queries.shape[0] * keys.shape[0] * D / (t * 1e-3) / 1e12, 2)}
    del q64, k64, out
    torch.cuda.empty_cache()
    return res


def baseline(queries, keys, k, exact_index, reps):
    def run():
        return torch.topk(F.normalize(queries, dim=1) @ F.normalize(keys, dim=1).t(), k, dim=1).indices
    t, idx = host_ms(run, reps)
    differ = sum(len(set(a) - set(b)) for a, b in zip(idx.tolist(), exact_index.tolist()))
    return {"baseline_ms": round(t, 3), "baseline_topk_not_exact": differ, "baseline_topk_total": idx.numel()}


def workload(name, keys, Q, seps, k, reps, device, windows=None):
    g = torch.Generator(device=device).manual_seed(Q)
    rows = torch.randint(0, keys.shape[0], (Q,), generator=g, device=device)
    queries = (keys[rows] + torch.randn(Q, D, generator=g, device=device)).contiguous()
    res = []
    for sep in seps:
        r = {"workload": name, "keys": keys.shape[0], "queries": Q, "separation_samples": sep,
             "keys_mb": round(keys.numel() * 4 / 2 ** 20, 1),
             # keys and score block together within the 126 MB L2: the kernel times are L2-resident
             "l2_resident": keys.numel() * 4 + Q * keys.shape[0] * 4 <= 126e6}
        ranges = None
        if sep:
            ranges = search._stage(search.neighbour_ranges(windows["recording"].cpu().numpy(),
                                                           windows["start"].cpu().numpy(), sep), device)
        r.update(kernels(queries, keys, ranges, min(k, keys.shape[0]), reps))
        t, out = host_ms(lambda: search.search(queries, windows if windows is not None else keys, k,
                                               separation_samples=sep), reps)
        r["search_ms"] = round(t, 3)
        r["hits_per_query"] = round((out["index"] >= 0).sum().item() / Q, 2)
        if sep == 0:
            r.update(mm_f64(queries, keys, reps))
            r["scoring_over_mm_f64"] = round(r["mm_f64_ms"] / r["cosine_scores_ms"], 3)
            r.update(baseline(queries, keys, k, out["index"], reps))
        print(json.dumps(r), file=sys.stderr, flush=True)
        res.append(r)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", default="1,100,1000")
    ap.add_argument("--library", type=int, default=1_000_000)
    ap.add_argument("--k", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--device", default="cuda:0")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_search.py measures the GPU: no CUDA device found")
    device = torch.device(args.device)
    torch.cuda.set_device(device)
    results = []
    for hours in (1, 24):
        n = hours * 3600
        keys = embeddings(n, hours, device)
        start = torch.arange(n, dtype=torch.int64, device=device) * HOP
        win = {"scene_embeddings": keys, "recording": torch.zeros(n, dtype=torch.int64, device=device),
               "start": start, "length": torch.full((n,), W, dtype=torch.int64, device=device)}
        for Q in (int(x) for x in args.queries.split(",") if x):
            results += workload(f"{hours}h", keys, Q, (0, W, HOUR), args.k, args.reps, device, win)
        del keys, win
        torch.cuda.empty_cache()
    if args.library:
        keys = embeddings(args.library, 7, device)
        results += workload("library", keys, 1000, (0,), args.k, args.reps, device)
    print(json.dumps({"gpu": gpu_info(device.index or 0), "dims": D, "k": args.k, "results": results}))


if __name__ == "__main__":
    main()
