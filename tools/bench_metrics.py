"""Tagging metrics on the GPU: what metrics.tagging_metrics and its kernels cost at AudioSet's shapes, next to sklearn on
the host, and how the chunk size METRICS_BLOCK_BYTES sets the time at 2 M clips.

  python tools/bench_metrics.py [--sizes 20371,2000000] [--reps 5] [--sklearn-classes 527]

Prints one JSON line with the GPU's name and power limit (read in the same run) and the host's CPU model and thread
count.  Inputs, K = 527 classes: scores are the sigmoid of seeded fp32 logits, targets follow a per-class prevalence
spread log-uniformly over [0.05 %, 20 %] (AudioSet's is skewed like that) with one positive and one negative forced
per class, and a positive's logit is shifted up by 2 so the metrics are not those of noise.  Inputs stay on the device.

  metrics_ms     metrics.tagging_metrics end to end (checks, chunks, copy back, final divisions): CUDA events around
                 --reps calls after a warm-up, per call
  kernels_ms     the acx_tagging_metrics launches alone over all chunks, same method
  chunks         at N = 2 M also kernels_ms for several METRICS_BLOCK_BYTES (classes per chunk kc): with the default
                 kc = 128 fewer blocks than SMs run at a time
  sklearn_s      average_precision_score + roc_auc_score (average=None) on the host at N = 20 371 over
                 --sklearn-classes classes; at N = 2 M over 8 classes only, reported per class
  check          the device counts equal metrics.reference_counts on 8 classes at every size"""
import argparse
import json
import os
import platform
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from audioset_convnext_inf_b200 import _native, metrics   # noqa: E402
from bench_windows import gpu_info                         # noqa: E402

K = 527


def inputs(N, device, seed):
    g = torch.Generator(device=device).manual_seed(seed)
    prevalence = 10 ** torch.empty(K, device=device).uniform_(-3.3, -0.7, generator=g)
    targets = (torch.rand(N, K, generator=g, device=device) < prevalence).to(torch.uint8)
    targets[0] = 1
    if N > 1:
        targets[1] = 0
    logits = torch.randn(N, K, generator=g, device=device) * 1.5 - 3.0 + 2.0 * targets
    return torch.sigmoid(logits), targets


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


def kernels(scores, targets, block_bytes, reps):
    N = scores.shape[0]
    kc = min(K, max(1, block_bytes // (16 * N)))
    ws = torch.empty(metrics.workspace_bytes(N, kc), dtype=torch.uint8, device=scores.device)
    out = torch.empty(K, 4, dtype=torch.int64, device=scores.device)
    st = torch.cuda.current_stream().cuda_stream

    def run():
        for c0 in range(0, K, kc):
            _native.call("acx_tagging_metrics", scores.data_ptr(), N, K, c0, min(kc, K - c0), targets.data_ptr(),
                         ws.data_ptr(), out[c0].data_ptr(), st)

    t = gpu_ms(run, reps)
    res = {"block_bytes": block_bytes, "kc": kc, "workspace_gb": round(ws.numel() / 1e9, 2), "kernels_ms": round(t, 3)}
    del ws
    torch.cuda.empty_cache()
    return res, out.cpu().numpy().view(np.uint64)


def sklearn_s(scores, targets):
    from sklearn import metrics as skm
    s, t = scores.cpu().numpy(), targets.cpu().numpy()
    t0 = time.perf_counter()
    ap = skm.average_precision_score(t, s, average=None)
    t1 = time.perf_counter()
    auc = skm.roc_auc_score(t, s, average=None)
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1, ap, auc


def cpu_info():
    model = platform.processor()
    try:
        with open("/proc/cpuinfo") as fh:
            model = next(line.split(":", 1)[1].strip() for line in fh if line.startswith("model name"))
    except (OSError, StopIteration):
        pass
    return {"model": model, "threads": os.cpu_count(), "torch_threads": torch.get_num_threads()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="20371,2000000")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sklearn-classes", type=int, default=K)
    ap.add_argument("--device", default="cuda:0")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_metrics.py measures the GPU: no CUDA device found")
    device = torch.device(args.device)
    torch.cuda.set_device(device)
    results = []
    for N in (int(x) for x in args.sizes.split(",") if x):
        scores, targets = inputs(N, device, N)
        r = {"clips": N, "classes": K, "scores_mb": round(N * K * 4 / 2 ** 20, 1)}
        r["metrics_ms"] = round(gpu_ms(lambda: metrics.tagging_metrics(scores, targets), args.reps), 3)
        res, counts = kernels(scores, targets, metrics.METRICS_BLOCK_BYTES, args.reps)
        r.update(res)
        cols = np.linspace(0, K - 1, 8).astype(int)
        want = metrics.reference_counts(scores[:, cols].cpu().numpy(), targets[:, cols].cpu().numpy())
        r["check_classes"] = cols.tolist()
        r["check_equal"] = bool(np.array_equal(counts[cols], want))
        got = metrics.tagging_metrics(scores, targets)
        r["mAP"] = round(float(got["average_precision"].mean()), 6)
        r["mean_auc"] = round(float(got["auc"].mean()), 6)
        if N >= 1_000_000:
            r["chunks"] = [kernels(scores, targets, b, max(1, args.reps // 2))[0]
                           for b in (1 << 30, 4 << 30, 16 << 30, 16 * N * K + 4096 * K)]
            c8 = slice(0, 8)
            t_ap, t_auc, _, _ = sklearn_s(scores[:, c8], targets[:, c8])
            r["sklearn_8_classes_s"] = {"ap": round(t_ap, 3), "auc": round(t_auc, 3),
                                        "per_class": round((t_ap + t_auc) / 8, 3)}
        else:
            kk = min(K, args.sklearn_classes)
            t_ap, t_auc, sap, sauc = sklearn_s(scores[:, :kk], targets[:, :kk])
            r["sklearn_s"] = {"classes": kk, "ap": round(t_ap, 3), "auc": round(t_auc, 3)}
            r["max_abs_diff_vs_sklearn"] = {"ap": float(np.abs(got["average_precision"][:kk] - sap).max()),
                                            "auc": float(np.abs(got["auc"][:kk] - sauc).max())}
        print(json.dumps(r), file=sys.stderr, flush=True)
        results.append(r)
        del scores, targets
        torch.cuda.empty_cache()
    print(json.dumps({"gpu": gpu_info(device.index or 0), "cpu": cpu_info(), "results": results}))


if __name__ == "__main__":
    main()
