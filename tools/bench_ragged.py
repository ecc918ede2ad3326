"""Ragged batches on the GPU: what batching clips of different lengths buys, and what the per-clip bounds cost.

  python tools/bench_ragged.py [--clips 512] [--reps 3] [--overhead-iters 20]

Prints one JSON line with the GPU's name and power limit (read in the same run) and two legs:

  throughput  `--clips` seeded clips with lengths uniform in 15-30 s (the range of Clotho, which
              pytorch/extract_embeddings.py loops over), white noise x 0.1 clamped to [-1, 1], bf16 mode, the
              reference's random init.  The exact-length path (every distinct length is its own batch, i.e. one
              forward_all per clip on such a list) against extract.extract_clipwise (length-sorted ragged batches),
              alternating in one process, host lists in and host results out on both sides.  Reports clips/s, seconds
              of audio per second, the sample-weighted padding fraction of the ragged canvases, and whether both
              paths returned identical logits.
  overhead    64 clips of exactly 320 000 samples, CUDA graphs on: forward_all(x) against
              forward_all(x, lengths=[320000] * 64), alternating -- the cost of the masked kernels when nothing is masked.

Every timed window ends in a device synchronise, and every shape it uses is run once before timing."""
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
from audioset_convnext_inf_b200.extract import extract_clipwise, length_buckets, ragged_batches   # noqa: E402

SR = 32000


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


def exact_length_path(model, waveforms, max_batch=64, want=("clipwise_logits",)):
    """The extraction before ragged batches: one batch per exact length (extract.length_buckets)."""
    dev = next(model.parameters()).device
    res = {k: [None] * len(waveforms) for k in want}
    for n, idx in length_buckets([len(w) for w in waveforms], max_batch):
        batch = torch.stack([torch.as_tensor(waveforms[i]) for i in idx]).to(dev)
        with torch.no_grad():
            out = model.forward_all(batch)
        for k in want:
            host = out[k].float().cpu()
            for j, i in enumerate(idx):
                res[k][i] = host[j]
    return res


def timed(fn, device):
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize(device)
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=512)
    ap.add_argument("--reps", type=int, default=3, help="alternations of the throughput leg")
    ap.add_argument("--overhead-iters", type=int, default=20, help="forwards per timed window of the overhead leg")
    ap.add_argument("--overhead-reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--device", default="cuda:0")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ragged.py measures the GPU: no CUDA device found")
    device = torch.device(args.device)
    torch.cuda.set_device(device)
    torch.manual_seed(0)       # the reference's own random init (convnext.py:263-267, 705-706), as bench.py
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
    m = m.to(device).eval().set_precision("bf16")

    # ---- throughput: 15-30 s clips -------------------------------------------------------------------------------
    rng = np.random.default_rng(args.seed)
    lengths = rng.integers(15 * SR, 30 * SR + 1, size=args.clips).tolist()
    waves = [np.clip(rng.standard_normal(n, dtype=np.float32) * 0.1, -1.0, 1.0) for n in lengths]
    plan = ragged_batches(lengths, 64)
    canvas_samples = sum(c * len(idx) for c, idx in plan)
    audio_s = sum(lengths) / SR
    ref, new = exact_length_path(m, waves), extract_clipwise(m, waves)         # warm-up: every shape of both paths
    identical = all(torch.equal(a, b) for a, b in zip(ref["clipwise_logits"], new["clipwise_logits"]))
    t_exact, t_ragged = [], []
    for _ in range(args.reps):
        t_exact.append(timed(lambda: exact_length_path(m, waves), device)[0])
        t_ragged.append(timed(lambda: extract_clipwise(m, waves), device)[0])
    te, tr = statistics.median(t_exact), statistics.median(t_ragged)
    throughput = {
        "clips": args.clips, "audio_s": round(audio_s, 1), "distinct_lengths": len(set(lengths)),
        "ragged_batches": len(plan), "padding_fraction": round(1.0 - sum(lengths) / canvas_samples, 4),
        "exact_length": {"s": [round(t, 4) for t in t_exact], "clips_per_s": round(args.clips / te, 1),
                         "audio_s_per_s": round(audio_s / te, 1)},
        "ragged": {"s": [round(t, 4) for t in t_ragged], "clips_per_s": round(args.clips / tr, 1),
                   "audio_s_per_s": round(audio_s / tr, 1)},
        "speedup": round(te / tr, 2), "identical_logits": identical}
    del waves, ref, new

    # ---- overhead: the masked kernels on a uniform batch ---------------------------------------------------------
    g = torch.Generator().manual_seed(args.seed + 1)
    x = (torch.randn(64, 10 * SR, generator=g) * 0.1).clamp_(-1.0, 1.0).to(device)
    full = [10 * SR] * 64
    with torch.no_grad():
        for _ in range(3):                          # graphs are captured on a shape's second use
            m.forward_all(x)
            m.forward_all(x, lengths=full)
        a, b = m.forward_all(x), m.forward_all(x, lengths=full)
        same = all(torch.equal(a[k], b[k]) for k in ("clipwise_logits", "scene_embeddings", "frame_embeddings"))
        t_plain, t_masked = [], []
        for _ in range(args.overhead_reps):
            t_plain.append(timed(lambda: [m.forward_all(x) for _ in range(args.overhead_iters)], device)[0])
            t_masked.append(timed(lambda: [m.forward_all(x, lengths=full) for _ in range(args.overhead_iters)], device)[0])
    per = lambda ts: [round(1e3 * t / args.overhead_iters, 3) for t in ts]          # noqa: E731
    mp, mm = statistics.median(per(t_plain)), statistics.median(per(t_masked))
    overhead = {"batch": 64, "samples": 10 * SR, "plain_ms": per(t_plain), "ragged_ms": per(t_masked),
                "plain_median_ms": mp, "ragged_median_ms": mm, "overhead_pct": round(100.0 * (mm / mp - 1.0), 2),
                "identical_outputs": same}
    print(json.dumps({"gpu": gpu_info(device.index or 0), "throughput": throughput, "overhead": overhead}))


if __name__ == "__main__":
    main()
