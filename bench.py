#!/usr/bin/env python
"""Headline benchmark: clips/s of the audio-tagging forward (10 s @ 32 kHz clips, bf16 tensor-core mode).

  python bench.py --gpus N --steps K --warmup W            our arm (libacx kernels on B200)
  python bench.py --impl reference --gpus N ...             the reference's CPU path (oracle port) on host cores
  torchrun ... bench.py --gpus N ...                        N > 1: one rank per GPU, clips sharded by clip
  python bench.py ... --dump-outputs DIR                    also save the last timed step's outputs as DIR/<name>.npy

One step = one forward of BASELINE.json configs[1] (batch 64 synthetic clips, ConvNeXt-Tiny random init) per GPU
(weak scaling) followed, for N > 1, by the NCCL all-gather of the logits.  Prints ONE JSON line (rank 0).
Weights and inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CLIP_SAMPLES = 320000
BATCH = 64
N_ROTATE = 3            # 3 x 82 MB of input + ~0.5 GB of activations per chunk >> 126 MB L2


ROOFLINE_NOTES = {
    "mlp_fused": "fused pwconv1 -> GELU -> pwconv2 -> layer-scale -> residual; in the group-planar stages the kernel also "
                 "computes the per-row LayerNorm statistics and applies the LayerNorm as a rank-1 epilogue correction, work "
                 "that is not in the 16 M C^2 FLOP numerator; bound by GELU-epilogue instruction issue, not by the MMAs",
    "dwconv_ln": "49 fp32 FMA per element on the CUDA cores: its practical roof is the FP32 pipe (~37% of the HBM figure "
                 "at 100% FMA issue), see DESIGN.md",
    "dwconv_tc": "banded-Toeplitz tcgen05 GEMMs (M64 N32 K16); the MMAs stream their operands out of shared memory at "
                 "128 B/clk, which bounds the kernel at ~0.06 ms per stage-0 layer; numerator = 2 M C 2 B of HBM traffic",
}


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor_burst=d["bf16_tflops"], tensor_sust=d["bf16_tflops_sustained"],
                    source="measured")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor_sust=1400.0, source="fallback")   # B200_PROFILING.md


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.t.join(timeout=2)

    def mark(self):
        return len(self.rows)

    def summary(self, lo=0, hi=None):
        rows = self.rows[lo:hi]
        where = "timed region"
        if len([r for r in rows if len(r) == 6 and r[0].isdigit()]) < 2:
            rows, where = self.rows[lo:], "timed region + e2e region (timed region shorter than two samples)"
        ok = [r for r in rows if len(r) == 6 and r[0].isdigit()]
        if not ok:
            return None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in ok)]
        return {"sm_mhz": statistics.median(int(r[0]) for r in ok), "sm_max_mhz": int(ok[0][1]),
                "reasons": reasons, "samples": len(ok), "window": where}


def build_model(device):
    import audioset_convnext_inf_b200 as acx
    torch.manual_seed(0)   # the reference's own random init (convnext.py:263-267, 705-706)
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
    return m.to(device).eval().set_precision("bf16")


def synth_clips(batch, seed, device="cpu", pin=False):
    g = torch.Generator().manual_seed(seed)
    w = (torch.randn(batch, CLIP_SAMPLES, generator=g) * 0.1).clamp_(-1.0, 1.0)
    if pin:
        w = w.pin_memory()
    return w.to(device) if device != "cpu" else w


def cpu_reference_clips_per_s(state_dict, clips, iters, threads):
    """The reference's CPU path: oracle port (same ATen ops as convnext.py:287-331), fp32, all host threads."""
    from oracle import convnext_oracle as O
    torch.set_num_threads(threads)
    sd = {k: v.detach().cpu() for k, v in state_dict.items()}
    wave = synth_clips(clips, 123)
    with torch.no_grad():
        O.forward(wave[:1], sd)                       # warm-up
        t0 = time.perf_counter()
        for _ in range(iters):
            O.forward(wave, sd)
        dt = time.perf_counter() - t0
    return clips * iters / dt, dt


def _time_ms(fn, iters, device):
    """Median device time of fn() over `iters` runs (CUDA events, sync both sides)."""
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(device)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize(device)
        ts.append(e0.elapsed_time(e1))
    return statistics.median(ts)


def extras_single_gpu(model, eng, device, peaks):
    """The other BASELINE.json configs, measured in the same run (rank 0, one GPU):
    configs[2] front end only at batch 512, configs[0] batch-1 latency, configs[4] batch sweep 1..2048,
    plus the same-GPU comparator: the reference's ops in stock eager PyTorch (cuDNN / cuBLAS) on this B200."""
    out = {}
    g = torch.Generator(device=device).manual_seed(77)

    def clips(b):
        return (torch.randn(b, CLIP_SAMPLES, device=device, generator=g) * 0.1).clamp_(-1.0, 1.0)

    # ---- configs[2]: front end only, 512 clips --------------------------------------------------------------------
    w512 = clips(512)
    eng.run(w512[:64], want=("logmel",))
    eng.run(w512, want=("logmel",))
    api_ms = _time_ms(lambda: eng.run(w512, want=("logmel",)), 5, device)
    eng.start_timing(None)
    eng.run(w512, want=("logmel",))
    kern = {}
    for tag, ms in eng.stop_timing():
        kern[tag] = kern.get(tag, 0.0) + ms
    k_ms = sum(kern.values())
    T = CLIP_SAMPLES // 320 + 1
    bytes_alg = 512 * (CLIP_SAMPLES * 4.0 + T * 224 * 4.0)          # fp32 waveform in, fp32 log-mel out (as built)
    flops = 512 * T * 2.0 * (1024 * 2 * 513 + 513 * 224)
    out["frontend_only"] = {
        "workload": "STFT(1024, hop 320) + 224-bin log-mel + bn0, 512 synthetic 10 s clips (BASELINE.json configs[2])",
        "clips_per_s_kernels": round(512 / (k_ms * 1e-3), 1), "kernels_ms": {k: round(v, 4) for k, v in kern.items()},
        "clips_per_s_api": round(512 / (api_ms * 1e-3), 1), "api_ms": round(api_ms, 3),
        "api_note": "Engine.run(want=('logmel',)) also copies each chunk's log-mel into the caller's tensor",
        "hbm_gbs": round(bytes_alg / (k_ms * 1e-3) / 1e9, 1), "hbm_frac": round(bytes_alg / (k_ms * 1e-3) / 1e9 / peaks["hbm"], 4),
        "tflops_dense_dft": round(flops / (k_ms * 1e-3) / 1e12, 1),
        "tensor_frac": round(flops / (k_ms * 1e-3) / 1e12 / peaks["tensor_sust"], 4)}
    # the same config through the opt-in front end on folded frames (ACX_FRONTEND=folded; DESIGN.md k2): information only
    try:
        from audioset_convnext_inf_b200.engine import Engine
        eng_f = Engine(model.state_dict(), device, precision="bf16", frontend="folded")
        if eng_f.frontend == "folded":
            eng_f.run(w512[:64], want=("logmel",))
            eng_f.run(w512, want=("logmel",))
            eng_f.start_timing(None)
            eng_f.run(w512, want=("logmel",))
            kf = {}
            for tag, ms in eng_f.stop_timing():
                kf[tag] = kf.get(tag, 0.0) + ms
            kf_ms = sum(kf.values())
            out["frontend_only"]["folded_opt_in"] = {
                "clips_per_s_kernels": round(512 / (kf_ms * 1e-3), 1), "kernels_ms": {k: round(v, 4) for k, v in kf.items()},
                "note": "real-input symmetry of the windowed DFT: half the MMAs; not the default (log-mel accuracy on tonal audio)"}
        del eng_f
    except Exception as e:  # noqa: BLE001 -- an information leg must not take the bench line down
        out["frontend_only"]["folded_opt_in"] = {"error": str(e)[:200]}
    del w512
    torch.cuda.empty_cache()

    # ---- configs[0] / configs[4]: batch-1 latency and the batch sweep (tagging + scene embedding) --------------------
    sweep = []
    for b in (1, 8, 64, 256, 1024, 2048):
        w = clips(b)
        for _ in range(3):
            eng.run(w, want=("logits", "scene"))
        ms = _time_ms(lambda: eng.run(w, want=("logits", "scene")), 20 if b <= 64 else 3, device)
        sweep.append({"batch": b, "ms": round(ms, 4), "clips_per_s": round(b / (ms * 1e-3), 1)})
        del w
    out["latency_b1"] = {"ms": sweep[0]["ms"], "workload": "one 10 s clip, tagging + scene embedding, CUDA-graph replay "
                         "(BASELINE.json configs[0] shape on the GPU)"}
    out["sweep"] = {"workload": "tagging + scene embeddings, device-resident synthetic clips (BASELINE.json configs[4])",
                    "points": sweep}

    # ---- same-GPU comparator: the reference's own ops, stock eager PyTorch on this B200 -----------------------------
    from oracle import convnext_oracle as O
    sd = {k: v.detach().to(device) for k, v in model.state_dict().items()}
    w = clips(BATCH)
    eager = {}
    with torch.no_grad(), O.on_device(device):
        def fp32():
            return O.forward(w, sd)

        def amp():
            lm = O.frontend(w, sd)                                   # front end kept fp32 (bf16 DFT is 35 dB off)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                emb = O.forward_features(lm[:, None], sd)
                return torch.nn.functional.linear(emb, sd["head_audioset.weight"], sd["head_audioset.bias"])
        for name, fn in (("fp32", fp32), ("bf16_autocast", amp)):
            try:
                fn()
                fn()
                ms = _time_ms(fn, 5, device)
                eager[name] = {"ms_per_64_clips": round(ms, 3), "clips_per_s": round(BATCH / (ms * 1e-3), 1)}
            except Exception as e:  # noqa: BLE001 -- a measurement leg must not take the bench line down
                eager[name] = {"error": repr(e)[:200]}
    eager["what"] = ("oracle restatement of convnext.py:287-331 (F.conv1d DFT, matmul mel, F.conv2d, F.layer_norm, F.linear, "
                     "F.gelu) run eagerly on cuda: cuDNN / cuBLAS kernels, NCHW<->NHWC permutes as in the reference; "
                     f"allow_tf32 matmul={torch.backends.cuda.matmul.allow_tf32} cudnn={torch.backends.cudnn.allow_tf32}")
    out["gpu_eager_baseline"] = eager
    torch.cuda.empty_cache()
    return out


def extras_multi_gpu(model, eng, device, world, dist):
    """BASELINE.json configs[3]: forward_frame_embeddings on 128 clips per GPU (1024 at 8 GPUs) + all-gather of the
    768 x 31 x 7 outputs (85 MB per rank), serial and overlapped (chunk i's all-gather on a side stream under chunk
    i+1's kernels).  Device-timed, max over ranks."""
    per = 128
    g = torch.Generator(device=device).manual_seed(99 + dist.get_rank())
    w = (torch.randn(per, CLIP_SAMPLES, device=device, generator=g) * 0.1).clamp_(-1.0, 1.0)
    gathered = torch.empty(world * per, 768, 31, 7, device=device)
    side = torch.cuda.Stream(device=device)

    def compute_only():
        return eng.run(w, want=("frame",))["frame"]

    def serial():
        f = eng.run(w, want=("frame",))["frame"]
        dist.all_gather_into_tensor(gathered, f)

    chunks = [w[i:i + 64] for i in range(0, per, 64)]
    gath_c = [torch.empty(world * 64, 768, 31, 7, device=device) for _ in chunks]

    def overlapped():
        evs = []
        for c, gc in zip(chunks, gath_c):
            f = eng.run(c, want=("frame",))["frame"]
            ev = torch.cuda.Event()
            ev.record()
            with torch.cuda.stream(side):
                side.wait_event(ev)
                f.record_stream(side)
                dist.all_gather_into_tensor(gc, f)
            evs.append(f)
        torch.cuda.current_stream(device).wait_stream(side)

    def gather_only():
        dist.all_gather_into_tensor(gathered, frame)

    res = {}
    frame = compute_only()
    for name, fn in (("compute_only", compute_only), ("all_gather_only", gather_only), ("serial", serial),
                     ("overlapped", overlapped)):
        for _ in range(2):
            fn()
        dist.barrier()
        ms = torch.tensor([_time_ms(fn, 5, device)], device=device)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        res[name + "_ms"] = round(ms.item(), 3)
    bytes_rank = per * 768 * 31 * 7 * 4
    res.update({"workload": f"forward_frame_embeddings, {per} clips per GPU ({world * per} clips), all_gather_into_tensor of "
                            "(128, 768, 31, 7) fp32 per rank (BASELINE.json configs[3])",
                "bytes_per_rank": bytes_rank, "clips_per_s_serial": round(world * per / (res["serial_ms"] * 1e-3), 1),
                "clips_per_s_overlapped": round(world * per / (res["overlapped_ms"] * 1e-3), 1),
                "all_gather_busbw_gbs": round(bytes_rank * (world - 1) / (res["all_gather_only_ms"] * 1e-3) / 1e9, 1)})
    return res


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import audioset_convnext_inf_b200 as acx
    torch.manual_seed(0)
    sd = acx.convnext_tiny(drop_path_rate=0.0, after_stem_dim=[252, 56]).state_dict()
    threads = os.cpu_count() or 1
    from oracle import convnext_oracle as O
    torch.set_num_threads(threads)
    clips = 4                                          # bounded sample of the 64-clip step
    wave = synth_clips(clips, 123)
    sdc = {k: v.detach().cpu() for k, v in sd.items()}
    with torch.no_grad():
        for _ in range(max(1, min(args.warmup, 2))):
            O.forward(wave, sdc)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            O.forward(wave, sdc)
        dt = time.perf_counter() - t0
    v = clips * args.steps / dt
    sample = f"{args.steps} steps x {clips} of the {BATCH} clips of one step, fp32 torch CPU ops"
    print(json.dumps({
        "impl": "reference", "metric": "clips/sec (10s@32kHz, bf16)", "value": round(v, 3), "unit": "clips/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "audio tagging forward, batch 64 synthetic 10 s clips, ConvNeXt-Tiny (configs[1])",
                   "note": "reference CPU path = oracle port of convnext.py:287-331 (the Python reference cannot travel to the GPU box)"},
        "cpu_baseline": {"value": round(v, 3), "unit": "clips/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": round(v, 3), "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[0]/[2]/[3]/[4] and eager-GPU legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    model = build_model(device)
    eng = model._get_engine()
    inputs = [synth_clips(BATCH, 1000 * rank + i, device=device) for i in range(N_ROTATE)]
    gathered = torch.empty(world * BATCH, 527, device=device) if world > 1 else None

    def step(i):
        out = eng.run(inputs[i % N_ROTATE], want=("logits",))
        if world > 1:
            dist.all_gather_into_tensor(gathered, out["logits"])
        return out

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    clocks = ClockSampler(local_rank)
    clocks.__enter__()                   # started before the warm-up so nvidia-smi is already streaming when timing starts
    for i in range(args.warmup):
        step(i)
    fence()
    # untimed profiling pass: which kernel dominates the step?
    prof = eng.profile(inputs[0])
    by_tag = {}
    for tag, ms in prof:
        by_tag.setdefault(tag, []).append(ms)
    top = max(by_tag, key=lambda t: sum(by_tag[t]))
    fence()

    # ---- timed region: device-resident inputs, production path (CUDA-graph replay) ------------------------
    launches0 = eng.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence()
    mark0 = clocks.mark()
    e0.record()
    for i in range(args.steps):
        out = step(i)
    e1.record()
    fence()
    mark1 = clocks.mark()
    launches = eng.launches - launches0
    if args.dump_outputs and rank == 0:
        # written now: the passes below reuse `gathered`.  64 clips x (logits, probs, scene) is under 0.5 MB.
        dumped = {k: v.float().cpu().numpy() for k, v in out.items()}
        if world > 1:
            dumped["logits_all_ranks"] = gathered.float().cpu().numpy()
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    # ---- same K steps again with a CUDA-event pair around every launch of the dominant kernel (individual launches:
    #      events cannot bracket a node inside a replayed graph); used only for roofline.achieved ------------------
    eng.start_timing(only=top)
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    i0.record()
    for i in range(args.steps):
        step(i)
    i1.record()
    top_ms = [ms for _, ms in eng.stop_timing()]
    instr_total_ms = i0.elapsed_time(i1)
    ms = torch.tensor([e0.elapsed_time(e1)], device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = ms.item()
    value = world * BATCH * args.steps / (ms_total / 1e3)

    # ---- e2e: public API, pinned host inputs, H2D + forward + D2H of the result every step -------------
    # HostPipeline is the package's host-to-host entry point (the reference's eval loop, PU:88-137): batch i+1 is
    # copied H2D on a copy stream while batch i computes; every step's copies are inside the timed region.
    import audioset_convnext_inf_b200 as acx
    host = [synth_clips(BATCH, 5000 + 1000 * rank + i, pin=True) for i in range(3)]
    pipe = acx.HostPipeline(model, want=("logits",))
    pipe.run([host[i % 3] for i in range(3)])                  # warm-up
    fence()
    n_e2e = args.steps
    t0 = time.perf_counter()
    res = pipe.run([host[i % 3] for i in range(n_e2e)])
    if world > 1:
        dist.all_gather_into_tensor(gathered, res[-1]["logits"].to(device))
    fence()
    dt = torch.tensor([time.perf_counter() - t0], device=device)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    assert len(res) == n_e2e and res[0]["probs"].shape == (BATCH, 527)
    e2e_value = world * BATCH * n_e2e / dt.item()
    clocks.__exit__()
    extras = {}
    if not args.no_extras:
        if world > 1:
            extras["frame_allgather"] = extras_multi_gpu(model, eng, device, world, dist)
        elif rank == 0:
            extras = extras_single_gpu(model, eng, device, _peaks())

    if rank == 0:
        peaks = _peaks()
        n_chunk = min(eng.chunk, BATCH)
        bound, work = eng.algorithmic_work(top, n_chunk, CLIP_SAMPLES)
        avg_ms = sum(top_ms) / max(1, len(top_ms))
        if bound == "hbm":
            achieved, peak, unit = work / (avg_ms * 1e-3) / 1e9, peaks["hbm"], "GB/s"
        else:
            achieved, peak, unit = work / (avg_ms * 1e-3) / 1e12, peaks["tensor_sust"], "TFLOP/s"
        share = sum(top_ms) / instr_total_ms
        traffic = None            # dram read+write bytes per launch of that kernel, from the committed ncu capture
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.isfile(tpath):
            tj = json.load(open(tpath))
            if tj.get("clips_per_launch") == n_chunk:
                traffic = tj["bytes_per_launch"].get(top)
        # every kernel class of the step against its own roof (untimed per-kernel event pass, serialised launches)
        prof_total = sum(sum(v) for v in by_tag.values())
        all_kernels = []
        for tag, v in sorted(by_tag.items(), key=lambda kv: -sum(kv[1])):
            b, w = eng.algorithmic_work(tag, n_chunk, CLIP_SAMPLES)
            t = sum(v) / len(v) * 1e-3
            if w <= 0 or t <= 0:
                continue
            ach = w / t / (1e9 if b == "hbm" else 1e12)
            pk = peaks["hbm"] if b == "hbm" else peaks["tensor_sust"]
            all_kernels.append({"kernel": tag, "bound": b, "launches": len(v), "avg_launch_ms": round(t * 1e3, 4),
                                "achieved": round(ach, 1), "unit": "GB/s" if b == "hbm" else "TFLOP/s",
                                "frac": round(ach / pk, 3), "share_of_step": round(sum(v) / prof_total, 3)})
        res = {
            "metric": "clips/sec (10s@32kHz, bf16)", "value": round(value, 2), "unit": "clips/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_total / args.steps, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "audio tagging forward, batch 64 synthetic 10 s clips per GPU, ConvNeXt-Tiny random init "
                                   "(BASELINE.json configs[1])", "clips_per_step_per_gpu": BATCH, "clip_samples": CLIP_SAMPLES,
                       "chunk": eng.chunk, "frontend": eng.frontend, "mlp": eng.mlp,
                       "l2": f"inputs rotate over {N_ROTATE} batches (246 MB) and per-chunk activations (~0.5 GB) exceed the 126 MB L2",
                       "parallelism": f"dp{world} (clip-sharded replicas, all-gather of logits)"},
            "e2e": {"value": round(e2e_value, 2), "unit": "clips/s", "h2d_bytes_per_step": BATCH * CLIP_SAMPLES * 4,
                    "d2h_bytes_per_step": BATCH * (2 * 527 + 768) * 4, "steps": n_e2e,
                    "api": "HostPipeline(model).run(pinned fp32 host batches) -> host probs/logits; double-buffered H2D/D2H"},
            "gpu_launches": launches,
            "clocks": clocks.summary(mark0, mark1),
            "roofline": {"kernel": top, "bound": bound, "achieved": round(achieved, 2), "peak": peak, "unit": unit,
                         "frac": round(achieved / peak, 4), "traffic": traffic, "peak_source": peaks["source"] +
                         (" (sustained bf16 figure: kernel timed inside a long step)" if bound == "tensor" else " (copy)"),
                         "launches_timed": len(top_ms), "avg_launch_ms": round(avg_ms, 4),
                         "timed_in": "the same K steps repeated right after the timed region with individual launches "
                                     "(CUDA events cannot bracket a node of a replayed graph)",
                         "share_of_step": round(share, 4),
                         "note": ROOFLINE_NOTES.get(top.rsplit("_c", 1)[0], "")},
            "roofline_all": all_kernels,
        }
        res.update(extras)
        if not args.no_cpu_baseline and world == 1:
            threads = os.cpu_count() or 1
            # bounded sample: ~10-15 s of host work (about 240 clips at the ~20 clips/s of a 16-core box)
            v, secs = cpu_reference_clips_per_s(model.state_dict(), clips=8, iters=30, threads=threads)
            res["cpu_baseline"] = {"value": round(v, 3), "unit": "clips/s", "cores": threads, "kind": "port",
                                   "sample": f"30 x 8 clips of the 64-clip step ({secs:.1f} s), oracle port of the "
                                             "reference forward, fp32, torch CPU ops"}
        print(json.dumps(res))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
