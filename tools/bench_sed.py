"""Sound event detection on the GPU: what sed.detect costs next to the forward_windows call that produced its input, and
what detection adds to a live stream's push.

  python tools/bench_sed.py [--hours 1,24] [--streams 256,1024] [--seconds 18] [--timed 6]

Prints one JSON line with the GPU's name and power limit (read in the same run).  bf16 mode, the reference's random init,
10 s windows at a 1 s hop, bins of 1 s, merge gap 2 s, minimum duration 1 s; per-class thresholds are the 70 % / 50 %
quantiles of the first recording's own activity, so every class has events.  Audio is seeded noise (x 0.1, clamped to
[-1, 1]).

  recordings    per length: forward_windows time (one call, after a warm-up on a short recording), sed.detect time
                (median of 5 calls, host clock around the call and a device synchronise), their ratio, bins and events
  streams       per S: S streams of --seconds s fed 1 s pushes from pinned host memory, with and without detection; the
                median and p99 (with few pushes, the largest) of the last --timed pushes, each timed with a host clock
                around push() and a device synchronise, and the detection memory
  identical     every stream's activity rows and events from all calls equal sed.detect(forward_windows) of the same
                audio, bit for bit"""
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
from audioset_convnext_inf_b200 import sed   # noqa: E402
from bench_windows import gpu_info           # noqa: E402

W, HOP, SR = 320000, 32000, 32000


def timed(fn, device):
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize(device)
    return out, time.perf_counter() - t0


def noise(n, seed, device):
    g = torch.Generator(device=device).manual_seed(seed)
    return (torch.randn(n, generator=g, device=device) * 0.1).clamp_(-1, 1)


def detection_for(windows):
    act = sed.detect(windows, sed.Detection(SR, 1.0))["activity"]["activity"].double()
    on = torch.quantile(act, 0.7, dim=0).float().cpu().numpy()
    off = np.minimum(on, torch.quantile(act, 0.5, dim=0).float().cpu().numpy())
    return sed.Detection(SR, on, off, min_duration_samples=SR, merge_gap_samples=2 * SR)


def run_recording(m, hours, det, device):
    rec = noise(int(hours * 3600 * SR), 1, device)
    with torch.no_grad():
        win, t_win = timed(lambda: m.forward_windows(rec, W, HOP), device)
    times = []
    for _ in range(5):
        out, t = timed(lambda: sed.detect(win, det), device)
        times.append(t)
    t_sed = statistics.median(times)
    res = {"hours": hours, "windows": int(win["start"].numel()), "bins": int(out["activity"]["start"].numel()),
           "events": int(out["events"]["onset"].numel()), "forward_windows_s": round(t_win, 3),
           "detect_ms": round(1e3 * t_sed, 2), "detect_over_windows_pct": round(100 * t_sed / t_win, 3)}
    del rec, win, out
    torch.cuda.empty_cache()
    return res


def run_streams(m, S, seconds, timed_n, det, device):
    base = noise(7919 * S + seconds * SR, 2, device).cpu().pin_memory()
    recs = [base[7919 * i:7919 * i + seconds * SR] for i in range(S)]
    out = {"streams": S}
    for label, d in (("plain", None), ("detection", det)):
        s = m.open_stream(S, W, HOP, detection=d)
        lat, calls = [], []
        with torch.no_grad():
            for t in range(seconds):
                res, dt = timed(lambda: s.push([r[t * SR:(t + 1) * SR] for r in recs]), device)
                calls.append(res)
                lat.append(dt)
            calls.append(s.close())
        steady = lat[-timed_n:]
        out[label] = {"push_ms": {"median": round(1e3 * statistics.median(steady), 2),
                                  "p99": round(1e3 * float(np.percentile(steady, 99)), 2)},
                      "real_time": float(np.percentile(steady, 99)) < 1.0}
        if d is not None:
            out[label]["detection_mb"] = round(s.detection_bytes / 2 ** 20, 1)
            with torch.no_grad():
                ref = sed.detect(m.forward_windows(recs, W, HOP), d)
            act = {k: torch.cat([c["activity"][k] for c in calls]) for k in sed.ACTIVITY_KEYS}
            order = torch.from_numpy(np.argsort(act["recording"].cpu().numpy(), kind="stable")).to(device)
            same = all(torch.equal(act[k].index_select(0, order), ref["activity"][k]) for k in sed.ACTIVITY_KEYS)
            ev = {k: torch.cat([c["events"][k] for c in calls]) for k in sed.EVENT_KEYS}
            key = (ev["recording"].cpu().numpy() * 527 + ev["class"].cpu().numpy()) * 2 ** 36 + ev["onset"].cpu().numpy()
            order = torch.from_numpy(np.argsort(key, kind="stable")).to(device)
            same &= all(torch.equal(ev[k].index_select(0, order), ref["events"][k]) for k in sed.EVENT_KEYS)
            out["identical"] = bool(same)
            out["events"] = int(ev["onset"].numel())
        del s, calls
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hours", default="1,24")
    ap.add_argument("--streams", default="256,1024")
    ap.add_argument("--seconds", type=int, default=18, help="audio per stream, pushed 1 s at a time")
    ap.add_argument("--timed", type=int, default=6, help="steady-state pushes timed at the end of each stream")
    ap.add_argument("--device", default="cuda:0")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sed.py measures the GPU: no CUDA device found")
    if args.seconds < 12 or not 1 <= args.timed <= args.seconds - 11:
        raise SystemExit("--seconds must be at least 12 and --timed at most seconds - 11 (the first bin is final at 11 s)")
    device = torch.device(args.device)
    torch.cuda.set_device(device)
    torch.manual_seed(0)       # the reference's own random init (convnext.py:263-267, 705-706), as bench.py
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
    m = m.to(device).eval().set_precision("bf16")
    with torch.no_grad():
        det = detection_for(m.forward_windows(noise(120 * SR, 3, device), W, HOP))   # also warms up the graphs
    recordings = [run_recording(m, float(h), det, device) for h in args.hours.split(",") if h]
    for r in recordings:
        print(json.dumps(r), file=sys.stderr, flush=True)
    streams = []
    for S in (int(x) for x in args.streams.split(",") if x):
        streams.append(run_streams(m, S, args.seconds, args.timed, det, device))
        print(json.dumps(streams[-1]), file=sys.stderr, flush=True)
    print(json.dumps({"gpu": gpu_info(device.index or 0), "window": W, "hop": HOP, "resolution": SR,
                      "recordings": recordings, "streams": streams,
                      "identical": all(s.get("identical", False) for s in streams)}))


if __name__ == "__main__":
    main()
