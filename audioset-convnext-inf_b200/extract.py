"""Counterpart of the reference's per-file extraction loop (pytorch/extract_embeddings.py:64-92: one forward per wav,
whatever its length) for a LIST of variable-length clips (SURVEY §8 row f3).

The model's result for a clip depends on its exact length (reflect padding, frame count), so clips are never simply
zero-padded to a common length.  They run as RAGGED batches instead (ConvNeXt.forward_all(x, lengths=...)): clips of
similar length share a canvas, and every kernel bounds each clip by its own length.  The outputs are returned in the
caller's order -- identical to looping clip by clip, at batch throughput."""
import collections

import numpy as np
import torch

from . import preprocess
from .engine import MIN_RAGGED_LEN

CANVAS_STEP = 32000        # canvases are whole seconds: few distinct workspace shapes (and CUDA graphs) per clip list


def length_buckets(lengths, max_batch):
    """[(length, [indices...])...]: indices grouped by equal length, split into runs of at most max_batch."""
    by_len = collections.OrderedDict()
    for i, n in enumerate(lengths):
        by_len.setdefault(int(n), []).append(i)
    out = []
    for n, idx in by_len.items():
        for s in range(0, len(idx), max_batch):
            out.append((n, idx[s:s + max_batch]))
    return out


def ragged_batches(lengths, max_batch, step=CANVAS_STEP):
    """[(canvas, [indices...])...]: indices sorted by length (ties in input order), cut into runs of at most max_batch;
    each run's canvas is its longest length rounded up to a multiple of `step`."""
    order = sorted(range(len(lengths)), key=lambda i: (int(lengths[i]), i))
    out = []
    for s in range(0, len(order), max_batch):
        idx = order[s:s + max_batch]
        longest = max(int(lengths[i]) for i in idx)
        out.append(((longest + step - 1) // step * step, idx))
    return out


def extract_clipwise(model, waveforms, max_batch=64, want=("clipwise_logits",), sample_rate=32000):
    """waveforms: sequence of 1-D float arrays / tensors (any lengths) at `sample_rate`.  Returns {name: list of per-clip
    tensors on the host, in input order} for the names in `want` (keys of ConvNeXt.forward_all); a clip's
    "frame_embeddings" cover its own frames only, like a forward of that clip alone.

    sample_rate: the clips' rate in Hz, a positive int or one per clip (default 32 kHz, the model's rate).  Clips not at
    32 kHz are resampled on the GPU (preprocess.resample; int16 clips are then PCM, read as x / 32767) in one launch per
    rate into one device buffer, and the ragged canvases are filled from that buffer on the device.  The results equal
    extract_clipwise of the resampled clips, bit for bit.  A clip whose resampled length is under 7360 samples raises
    ValueError before anything is launched."""
    dev = next(model.parameters()).device
    rates = preprocess.sample_rates(sample_rate, len(waveforms))
    buf = None
    if any(r != preprocess.SAMPLE_RATE for r in rates):
        clips = preprocess.check_waveforms(
            [w if isinstance(w, torch.Tensor) else torch.from_numpy(np.asarray(w)) for w in waveforms], "clip")
        lengths = [preprocess.resampled_length(w.numel(), r) for w, r in zip(clips, rates)]
        for i, n in enumerate(lengths):
            if n < MIN_RAGGED_LEN:
                raise ValueError(f"clip {i} has {n} samples once resampled to 32 kHz; the shortest the model takes is "
                                 f"{MIN_RAGGED_LEN}")
        buf, _ = preprocess.resample_packed(clips, rates, preprocess.SAMPLE_RATE, dev)
        offsets = np.concatenate([[0], np.cumsum(lengths, dtype=np.int64)]).tolist()
    else:
        lengths = [len(w) for w in waveforms]
    res = {k: [None] * len(waveforms) for k in want}
    for canvas, idx in ragged_batches(lengths, max_batch):
        if buf is None:
            batch = torch.zeros(len(idx), canvas, dtype=torch.float32)
            for j, i in enumerate(idx):
                batch[j, :lengths[i]] = torch.as_tensor(np.asarray(waveforms[i]), dtype=torch.float32)
            batch = batch.to(dev)
        else:
            batch = torch.zeros(len(idx), canvas, dtype=torch.float32, device=dev)
            for j, i in enumerate(idx):
                batch[j, :lengths[i]] = buf[offsets[i]:offsets[i + 1]]
        with torch.no_grad():
            out = model.forward_all(batch, lengths=[lengths[i] for i in idx])
        frames = out["frame_lengths"].tolist()
        for k in want:
            host = out[k].cpu() if k == "frame_lengths" else out[k].float().cpu()
            for j, i in enumerate(idx):
                res[k][i] = host[j, :, :frames[j]] if k == "frame_embeddings" else host[j]
    return res
