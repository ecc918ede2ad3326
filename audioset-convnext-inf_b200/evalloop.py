"""Drop-in for the reference's batch inference loop `pytorch_utils.forward` (reference
src/audioset_convnext_inf/pytorch/pytorch_utils.py:63-137) and for its caller `Evaluator` (evaluate.py:12-60).

Same name, arguments, and return value (dict of concatenated numpy arrays), but the per-batch
`move_data_to_device` -> `model(batch)` -> `.data.cpu().numpy()` sequence runs through `HostPipeline`, so the H2D
copy of batch i+1 and the D2H copy of batch i-1 overlap the kernels of batch i.  Waveforms may be float32 or the
int16 PCM the AudioSet HDF5 files hold (data_generator.py:70-74).  `Evaluator.evaluate` scores the clipwise output
against the targets on the GPU (metrics.tagging_metrics) instead of with sklearn on the host.
"""
import numpy as np
import torch

from . import metrics
from .pipeline import HostPipeline


def _as_host_batch(w):
    if isinstance(w, torch.Tensor):
        t = w.detach().cpu()
    else:
        arr = np.asarray(w)
        if arr.dtype == object:        # the reference's collate_fn builds dtype=object arrays (data_generator.py:517-519)
            arr = np.stack([np.asarray(a) for a in arr])
        t = torch.from_numpy(np.ascontiguousarray(arr))
    if t.dtype not in (torch.float32, torch.int16):
        t = t.to(torch.float32)
    return t.contiguous()


def forward(model, generator, use_torchaudio=False, return_input=False, return_target=False):
    """See pytorch_utils.forward (PU:63-82).  Returns {"clipwise_output": (N, 527) [, "waveform", "target"]}."""
    if use_torchaudio:
        raise NotImplementedError("the torchaudio fbank front end (use_torchaudio=True) is out of scope")
    model.eval()
    inputs, targets = [], []

    def host_batches():
        # one batch at a time: the loader (HDF5 reads in the reference) overlaps with the kernels of the previous batch
        # and nothing but the pipeline's `depth` staging buffers is ever page-locked
        for batch_data_dict in generator:
            hb = _as_host_batch(batch_data_dict["waveform"])
            if return_input:
                inputs.append(hb.numpy())
            if return_target and "target" in batch_data_dict:
                targets.append(np.asarray(batch_data_dict["target"]))
            yield hb

    # batches of equal shape stream through one pipeline; a ragged last batch simply re-allocates its slots
    results = HostPipeline(model, want=("logits",)).run(host_batches())
    out = {"clipwise_output": np.concatenate([r["probs"].numpy() for r in results], axis=0)}
    if return_input:
        out["waveform"] = np.concatenate(inputs, axis=0)
    if return_target and targets:
        out["target"] = np.concatenate(targets, axis=0)
    return out


class Evaluator:
    """The reference's Evaluator (evaluate.py:12-60): Evaluator(model).evaluate(data_loader)."""

    def __init__(self, model):
        self.model = model

    def evaluate(self, data_loader):
        """forward(model, data_loader, return_target=True), then per-class metrics of the clipwise output against the
        targets on the model's device.  Returns {"average_precision", "auc", "d_prime"}, each a (classes,) float64
        numpy array.  Raises ValueError when the loader yields no "target"."""
        out = forward(self.model, data_loader, return_target=True)
        if "target" not in out:
            raise ValueError("the data loader yields no \"target\": there is nothing to score the clipwise output against")
        dev = next(self.model.parameters()).device
        stats = metrics.tagging_metrics(torch.from_numpy(out["clipwise_output"]).to(dev), out["target"])
        return {"average_precision": stats["average_precision"], "auc": stats["auc"],
                "d_prime": metrics.d_prime(stats["auc"])}
