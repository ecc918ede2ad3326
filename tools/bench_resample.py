"""Resampling long recordings to 32 kHz on the GPU: the segmented resampler against acx_resample_fit and torchaudio, and
its share of ConvNeXt.forward_windows(sample_rate=...).

  python tools/bench_resample.py [--hours 1] [--reps 5] [--rates 44100,48000] [--hops 320000,32000] [--no-torchaudio]

Prints one JSON line with the GPU's name and power limit (read in the same run).  Workload: one seeded recording of
`--hours` hours per rate (white noise x 0.1 clamped to [-1, 1]; its int16 form is round(x * 32767)), bf16 mode, the
reference's random init.  Per rate:

  kernel          acx_resample_segments(_pcm16) on the whole recording as one segment: CUDA events around each launch,
                  after a warm-up launch, `--reps` times (the 44.1 kHz hour's output is 460 MB and its input 635 MB, more
                  than L2, so every launch reads from HBM).  gfma_per_s counts out_len x K fused multiply-adds.
  fit             acx_resample_fit on the same hour as a (1, L) float32 batch at n_out = ceil(new L / orig), timed the same
                  way (it fits in 32-bit indices; int16 is converted x / 32767 first, outside the timing);
                  identical_to_fit compares the two outputs bit for bit.
  resample        preprocess.resample end to end (wall clock ending in a synchronise), from pinned host memory (the copy
                  to the device is inside) and from the device.
  windows         forward_windows(recording, 320000, hop, sample_rate=rate) from the device against forward_windows on the
                  already resampled 32 kHz buffer; resample_share = 1 - pre_resampled / with_resampling.  peak_mb is
                  torch.cuda.max_memory_allocated during one call above what was allocated before it (the model, the
                  recording).
  torchaudio      torchaudio.functional.resample of the float32 hour on the host (the status quo), once, and the largest
                  absolute difference from the GPU output on the common prefix (torchaudio may be one sample shorter)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import audioset_convnext_inf_b200 as acx                      # noqa: E402
from audioset_convnext_inf_b200 import _native, preprocess    # noqa: E402

SR = 32000
W = 10 * SR


def gpu_info(index):
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                            "-i", str(index)], capture_output=True, text=True, timeout=30)
        pl, mhz = (c.strip() for c in r.stdout.strip().split(","))
        info.update(power_limit_w=float(pl), sm_max_mhz=int(mhz))
    except (OSError, ValueError, subprocess.SubprocessError):
        info.update(power_limit_w=None, sm_max_mhz=None)
    return info


def event_times(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) / 1e3)
    return ts


def wall_times(fn, device, reps, warm=True):
    if warm:
        fn()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize(device)
        ts.append(time.perf_counter() - t0)
    return ts


def peak_mb(fn, device):
    torch.cuda.synchronize(device)
    start = torch.cuda.memory_allocated(device)
    torch.cuda.reset_peak_memory_stats(device)
    fn()
    torch.cuda.synchronize(device)
    return round((torch.cuda.max_memory_allocated(device) - start) / 2 ** 20, 1)


def summary(ts, **per_s):
    t = statistics.median(ts)
    out = {"s": [round(x, 5) for x in ts], "median_s": round(t, 5)}
    out.update({k: round(v / t, 1) for k, v in per_s.items()})
    return out


def kernel_launcher(x, rate, out, device):
    """A closure launching acx_resample_segments(_pcm16) on x as one segment into out (the table built once)."""
    taps, width, orig, new = preprocess._cached_taps(rate, SR, device)
    frames, groups = preprocess.segment_tiling(orig, new, width)
    start, n_tiles = preprocess.segment_tiles([out.numel()], frames, groups, new)
    table = torch.cat([torch.tensor([0, x.numel(), 0, out.numel()], dtype=torch.int64), start]).to(device)
    name = "acx_resample_segments_pcm16" if x.dtype == torch.int16 else "acx_resample_segments"
    stream = torch.cuda.current_stream(device).cuda_stream
    k = 2 * width + orig

    def run():
        _native.call(name, x.data_ptr(), x.numel(), table.data_ptr(), 1, table.data_ptr() + 32, n_tiles, taps.data_ptr(),
                     orig, new, width, out.data_ptr(), out.numel(), stream)
    return run, k


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hours", type=float, default=1.0)
    ap.add_argument("--rates", default="44100,48000")
    ap.add_argument("--hops", default=f"{W},{SR}", help="comma-separated hops in 32 kHz samples")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--no-torchaudio", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_resample.py measures the GPU: no CUDA device found")
    device = torch.device(args.device)
    torch.cuda.set_device(device)
    torch.manual_seed(0)       # the reference's own random init (convnext.py:263-267, 705-706), as bench.py
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
    m = m.to(device).eval().set_precision("bf16")
    hops = [int(h) for h in args.hops.split(",")]

    results = []
    for rate in (int(r) for r in args.rates.split(",")):
        n = int(args.hours * 3600 * rate)
        n_out = preprocess.resampled_length(n, rate)
        rng = np.random.default_rng(args.seed + rate)
        f32 = np.clip(rng.standard_normal(n, dtype=np.float32) * 0.1, -1.0, 1.0)
        recs = {"float32": torch.from_numpy(f32).pin_memory(),
                "int16": torch.from_numpy(np.round(f32 * 32767.0).astype(np.int16)).pin_memory()}
        del f32
        entry = {"rate": rate, "input_samples": n, "output_samples": n_out}
        gpu_out = None
        for dtype, host in recs.items():
            dev_rec = host.to(device)
            r = {}
            out = torch.empty(n_out, device=device)
            run, k = kernel_launcher(dev_rec, rate, out, device)
            r["kernel"] = summary(event_times(run, args.reps), out_samples_per_s=n_out, gfma_per_s=n_out * k / 1e9)
            r["kernel"]["taps"] = k
            xf = dev_rec if dev_rec.dtype == torch.float32 else \
                torch.div(dev_rec.float(), torch.tensor(32767.0, device=device))     # a true division, like the kernel's
            taps, width, orig, new = preprocess._cached_taps(rate, SR, device)
            fit_out = torch.empty(n_out, device=device)
            stream = torch.cuda.current_stream(device).cuda_stream

            def fit():
                _native.call("acx_resample_fit", xf.data_ptr(), n, taps.data_ptr(), fit_out.data_ptr(), n_out, 1, n,
                             orig, new, width, n_out, stream)
            r["fit"] = summary(event_times(fit, args.reps), out_samples_per_s=n_out, gfma_per_s=n_out * k / 1e9)
            r["identical_to_fit"] = bool(torch.equal(out, fit_out))
            r["kernel_speedup_over_fit"] = round(r["fit"]["median_s"] / r["kernel"]["median_s"], 2)
            del fit_out, xf
            if dtype == "float32":
                gpu_out = out.cpu()
            del out
            r["resample"] = {where: summary(wall_times(lambda: preprocess.resample(src, rate, device=device), device,
                                                       args.reps), audio_s_per_s=n / rate)
                             for where, src in (("host", host), ("device", dev_rec))}
            pre = preprocess.resample(dev_rec, rate)[0].clone()
            r["windows"] = {}
            for hop in hops:
                with torch.no_grad():
                    def with_rs():
                        return m.forward_windows(dev_rec, W, hop, sample_rate=rate)

                    def pre_rs():
                        return m.forward_windows(pre, W, hop)
                    a, b = with_rs(), pre_rs()
                    same = all(torch.equal(a[key], b[key]) for key in ("clipwise_logits", "scene_embeddings", "start"))
                    n_win = a["start"].numel()
                    del a, b
                    mem = {"with_resampling": peak_mb(with_rs, device), "pre_resampled": peak_mb(pre_rs, device)}
                    ts = {"with_resampling": [], "pre_resampled": []}
                    for _ in range(args.reps):                                 # alternate the two paths
                        ts["with_resampling"] += wall_times(with_rs, device, 1, warm=False)
                        ts["pre_resampled"] += wall_times(pre_rs, device, 1, warm=False)
                w = {key: dict(summary(v), peak_mb=mem[key]) for key, v in ts.items()}
                w["windows"] = n_win
                w["identical_outputs"] = same
                w["resample_share"] = round(1 - w["pre_resampled"]["median_s"] / w["with_resampling"]["median_s"], 4)
                r["windows"][hop] = w
            del pre, dev_rec
            torch.cuda.empty_cache()
            entry[dtype] = r
        if not args.no_torchaudio:
            import torchaudio.functional as TAF
            t0 = time.perf_counter()
            ref = TAF.resample(recs["float32"][None], rate, SR)[0]
            t = time.perf_counter() - t0
            c = min(ref.numel(), gpu_out.numel())
            entry["torchaudio_cpu"] = {"s": round(t, 3), "threads": torch.get_num_threads(),
                                       "audio_s_per_s": round(n / rate / t, 1), "samples": ref.numel(),
                                       "max_abs_diff_common_prefix": float((ref[:c] - gpu_out[:c]).abs().max())}
            del ref
        results.append(entry)
    print(json.dumps({"gpu": gpu_info(device.index or 0), "hours": args.hours, "results": results}))


if __name__ == "__main__":
    main()
