"""Live streams on the GPU: S streams fed 1 s pushes through ConvNeXt.open_stream, against one forward_windows call on the
same audio.

  python tools/bench_stream.py [--streams 64,256,1024] [--rates 32000,44100,48000] [--dtypes float32,int16] [--seconds 24]

Prints one JSON line with the GPU's name and power limit (read in the same run) and one entry per (S, rate, dtype).
Workload: S streams of `--seconds` s each, 10 s windows at a 1 s hop, bf16 mode, the reference's random init.  The audio is
one seeded noise signal (x 0.1, clamped to [-1, 1]; int16 is round(x * 32767)) in pinned host memory, stream i reading
it from offset 7919 i, so the streams differ.  Every push hands each stream the next second of its audio as a view of
that pinned buffer.  The first pushes fill the rings (no window is complete before 10 s) and capture the CUDA graphs;
the last `--timed` pushes, each timed with a host clock around push() and a device synchronise, are the steady state:

  push_ms         median and p99 (with few pushes, the largest) of one push, all S streams
  rtf             audio seconds tagged per wall second over the timed pushes (S x pushes / time)
  real_time       p99 push latency under 1 s: the S streams keep up with live audio
  ring_mb         device memory of the rings (fixed when the tagger is opened)
  stream_total_s  every push plus close, start to end of the stream
  windows_s       one forward_windows call on the same S recordings at the same rate (second of two calls)
  identical       the rows of all stream calls equal forward_windows' rows, bit for bit, for every key"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import audioset_convnext_inf_b200 as acx     # noqa: E402
from bench_windows import gpu_info           # noqa: E402

W, HOP = 320000, 32000
KEYS = ("clipwise_logits", "clipwise_output", "scene_embeddings", "recording", "start", "length")


def run_config(m, base, S, rate, seconds, timed_n, device):
    recs = [base[7919 * i:7919 * i + seconds * rate] for i in range(S)]
    s = m.open_stream(S, W, HOP, sample_rate=rate)
    lat, calls = [], []
    torch.cuda.synchronize(device)
    t_start = time.perf_counter()
    with torch.no_grad():
        for t in range(seconds):
            t0 = time.perf_counter()
            calls.append(s.push([r[t * rate:(t + 1) * rate] for r in recs]))
            torch.cuda.synchronize(device)
            lat.append(time.perf_counter() - t0)
        calls.append(s.close())
        torch.cuda.synchronize(device)
    stream_total = time.perf_counter() - t_start
    rows = {k: torch.cat([c[k] for c in calls]) for k in KEYS}
    order = torch.from_numpy(np.argsort(rows["recording"].cpu().numpy(), kind="stable")).to(device)
    rows = {k: v.index_select(0, order) for k, v in rows.items()}
    win_t = []
    with torch.no_grad():
        for _ in range(2):
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            ref = m.forward_windows(recs, W, HOP, sample_rate=rate)
            torch.cuda.synchronize(device)
            win_t.append(time.perf_counter() - t0)
    same = all(torch.equal(rows[k], ref[k]) for k in KEYS)
    steady = lat[-timed_n:]
    p99 = float(np.percentile(steady, 99))
    out = {"streams": S, "rate": rate, "dtype": str(base.dtype).replace("torch.", ""), "seconds": seconds,
           "windows": int(ref["length"].numel()), "timed_pushes": len(steady),
           "push_ms": {"median": round(1e3 * statistics.median(steady), 2), "p99": round(1e3 * p99, 2)},
           "rtf": round(S * len(steady) / sum(steady), 1), "real_time": p99 < 1.0,
           "ring_mb": round(s.ring_bytes / 2 ** 20, 1), "stream_total_s": round(stream_total, 3),
           "windows_s": round(win_t[-1], 3), "stream_over_windows": round(stream_total / win_t[-1], 3),
           "identical": same}
    del s, calls, rows, ref
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", default="64,256,1024")
    ap.add_argument("--rates", default="32000,44100,48000")
    ap.add_argument("--dtypes", default="float32,int16")
    ap.add_argument("--seconds", type=int, default=24, help="audio per stream, pushed 1 s at a time")
    ap.add_argument("--timed", type=int, default=12, help="steady-state pushes timed at the end of each stream")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--device", default="cuda:0")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stream.py measures the GPU: no CUDA device found")
    if args.seconds < 11 or not 1 <= args.timed <= args.seconds - 10:
        raise SystemExit("--seconds must be at least 11 and --timed at most seconds - 10 (the first window ends at 10 s)")
    device = torch.device(args.device)
    torch.cuda.set_device(device)
    torch.manual_seed(0)       # the reference's own random init (convnext.py:263-267, 705-706), as bench.py
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
    m = m.to(device).eval().set_precision("bf16")
    streams = [int(x) for x in args.streams.split(",")]
    rates = [int(x) for x in args.rates.split(",")]
    n = 7919 * max(streams) + args.seconds * max(rates)
    rng = np.random.default_rng(args.seed)
    f32 = np.clip(rng.standard_normal(n, dtype=np.float32) * 0.1, -1.0, 1.0)
    bases = {"float32": torch.from_numpy(f32), "int16": torch.from_numpy(np.round(f32 * 32767.0).astype(np.int16))}
    del f32
    results = []
    for dtype in args.dtypes.split(","):
        base = bases[dtype].pin_memory()
        for rate in rates:
            for S in streams:
                results.append(run_config(m, base, S, rate, args.seconds, args.timed, device))
                print(json.dumps(results[-1]), file=sys.stderr, flush=True)
        del base
    best = {}
    for r in results:
        if r["real_time"]:
            key = f'{r["rate"]}/{r["dtype"]}'
            best[key] = max(best.get(key, 0), r["streams"])
    print(json.dumps({"gpu": gpu_info(device.index or 0), "window": W, "hop": HOP, "largest_real_time_S": best,
                      "results": results}))


if __name__ == "__main__":
    main()
