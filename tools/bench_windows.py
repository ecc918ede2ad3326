"""Sliding windows over a long recording on the GPU: forward_windows (windows read in place) against materialised windows.

  python tools/bench_windows.py [--hours 1] [--reps 3] [--hops 320000,32000]

Prints one JSON line with the GPU's name and power limit (read in the same run) and one entry per (input dtype, hop,
input residence).  Workload: one seeded recording of `--hours` hours at 32 kHz (white noise x 0.1 clamped to [-1, 1]; its
int16 form is round(x * 32767)), 10 s windows, bf16 mode, the reference's random init.  Both paths compute clipwise
logits, probabilities and scene embeddings of the same window plan (windows.plan_windows):

  windows       ConvNeXt.forward_windows(recording, 320000, hop)
  materialised  the recording on the device, every window copied out (unfold(...).contiguous(), plus the end-aligned tail
                window when the hop grid leaves one), int16 converted x / 32767. first, then the engine call forward_all
                makes, without frame embeddings.

`host` inputs start in pinned host memory, so the host-to-device copy is inside the timed window (the recording itself on
both paths); `device` inputs are already on the GPU.  The two paths alternate in one process, every shape is run twice
before timing (a CUDA graph is captured on a shape's second use), and every timed window ends in a device synchronise.
peak_mb is torch.cuda.max_memory_allocated during one call, above what was allocated before it."""
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
from audioset_convnext_inf_b200.windows import plan_windows   # noqa: E402

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


def windows_path(model, rec, hop):
    with torch.no_grad():
        out = model.forward_windows(rec, W, hop)
    return out["clipwise_logits"], out["scene_embeddings"]


def materialised_path(model, rec, hop, device):
    eng = model._get_engine()
    x = rec.to(device, non_blocking=True)
    if x.dtype == torch.int16:
        x = torch.div(x.to(torch.float32), torch.tensor(32767.0, device=device))    # the prep kernels' x / 32767.
    n = x.numel()
    win = x.unfold(0, W, hop)
    if (win.shape[0] - 1) * hop + W < n:
        win = torch.cat([win, x[n - W:][None]])
    win = win.contiguous()
    del x
    out = eng.run(win, want=("logits", "scene"))
    return out["logits"], out["scene"]


def timed(fn, device):
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize(device)
    return time.perf_counter() - t0, out


def peak(fn, device):
    torch.cuda.synchronize(device)
    start = torch.cuda.memory_allocated(device)
    torch.cuda.reset_peak_memory_stats(device)
    out = fn()
    torch.cuda.synchronize(device)
    return (torch.cuda.max_memory_allocated(device) - start) / 2 ** 20, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hours", type=float, default=1.0)
    ap.add_argument("--hops", default=f"{W},{SR}", help="comma-separated hops in samples")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--device", default="cuda:0")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_windows.py measures the GPU: no CUDA device found")
    device = torch.device(args.device)
    torch.cuda.set_device(device)
    torch.manual_seed(0)       # the reference's own random init (convnext.py:263-267, 705-706), as bench.py
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
    m = m.to(device).eval().set_precision("bf16")

    n = int(args.hours * 3600 * SR)
    rng = np.random.default_rng(args.seed)
    f32 = np.clip(rng.standard_normal(n, dtype=np.float32) * 0.1, -1.0, 1.0)
    recs = {"float32": torch.from_numpy(f32).pin_memory(),
            "int16": torch.from_numpy(np.round(f32 * 32767.0).astype(np.int16)).pin_memory()}
    del f32
    results = []
    for dtype, host in recs.items():
        dev_rec = host.to(device)
        for hop in (int(h) for h in args.hops.split(",")):
            n_win = plan_windows([n], W, hop).length.numel()
            for where, rec in (("host", host), ("device", dev_rec)):
                paths = {"windows": lambda: windows_path(m, rec, hop),
                         "materialised": lambda: materialised_path(m, rec, hop, device)}
                outs = {k: [fn(), fn()][1] for k, fn in paths.items()}        # warm-up: graphs are captured on 2nd use
                same = all(torch.equal(a, b) for a, b in zip(outs["windows"], outs["materialised"]))
                del outs
                mem = {k: round(peak(fn, device)[0], 1) for k, fn in paths.items()}
                ts = {k: [] for k in paths}
                for _ in range(args.reps):
                    for k, fn in paths.items():
                        ts[k].append(timed(fn, device)[0])
                entry = {"dtype": dtype, "hop": hop, "input": where, "windows": n_win, "identical_outputs": same}
                for k in paths:
                    t = statistics.median(ts[k])
                    entry[k] = {"s": [round(x, 4) for x in ts[k]], "windows_per_s": round(n_win / t, 1),
                                "audio_s_per_s": round(n / SR / t, 1), "peak_mb": mem[k]}
                entry["speedup"] = round(statistics.median(ts["materialised"]) / statistics.median(ts["windows"]), 3)
                results.append(entry)
        del dev_rec
    print(json.dumps({"gpu": gpu_info(device.index or 0), "recording_s": n / SR, "window": W, "results": results}))


if __name__ == "__main__":
    main()
