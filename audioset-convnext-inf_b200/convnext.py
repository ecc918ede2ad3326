"""Drop-in mirror of the reference model API (reference: src/audioset_convnext_inf/pytorch/convnext.py).

Same class names, constructor arguments, parameter / buffer names and shapes (190-entry state dict,
28 222 767 trainable parameters), same three inference methods and return types:

    ConvNeXt.forward(x)                  -> {"clipwise_output": (B,527), "clipwise_logits": (B,527)}   CX:287-331
    ConvNeXt.forward_scene_embeddings(x) -> (B, 768)                                                   CX:333-366
    ConvNeXt.forward_frame_embeddings(x) -> (B, 768, T', 7)                                            CX:369-402
    ConvNeXt.from_pretrained(path_or_id) / convnext_tiny(...)                                          CX:404-511, 641-708

but nothing here computes with torch ops: the modules only hold parameters, and every forward
runs the hand-written sm_100a kernels of libacx.so through `engine.Engine`.  There is no CPU or
eager fallback -- calling a forward method on a non-CUDA model, or without libacx.so, raises.
Training-only behaviour of the reference (augmentations CX:288-295, SpecAugment CX:308-309, mixup
CX:312-313, DropPath) is out of scope and raises instead of silently differing.
"""
import os

import torch
import torch.nn as nn

from . import _native, preprocess
from .engine import DEPTHS, DIMS, Engine, out_time_dims
from .frontend_consts import slaney_mel_filterbank, windowed_dft
from .windows import plan_windows

HF_PYTORCH_WEIGHTS_NAME = "model.safetensors"
HF_CONFIG_NAME = "config.yaml"


class LayerNorm(nn.Module):
    """Parameter holder with the reference's dual-format signature (CX:514-541)."""

    def __init__(self, normalized_shape, eps=1e-6, data_format="channels_last"):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(normalized_shape))
        self.bias = nn.Parameter(torch.zeros(normalized_shape))
        self.eps = eps
        self.data_format = data_format
        if self.data_format not in ["channels_last", "channels_first"]:
            raise NotImplementedError
        self.normalized_shape = (normalized_shape,)

    def forward(self, x):
        raise RuntimeError("LayerNorm is fused into the libacx kernels; call the ConvNeXt forward methods")


class Block(nn.Module):
    """Parameter holder for one ConvNeXt block (CX:44-87): dwconv 7x7, LayerNorm, pwconv1, GELU,
    pwconv2, layer-scale gamma.  Computed by acx_dwconv_ln + acx_gemm_bf16 x2 (or acx_mlp_fused)."""

    def __init__(self, dim, drop_path=0.0, layer_scale_init_value=1e-6):
        super().__init__()
        if drop_path > 0.0:
            raise NotImplementedError("DropPath is training-only; the B200 path supports drop_path_rate=0.0")
        self.dwconv = nn.Conv2d(dim, dim, kernel_size=7, padding=3, groups=dim)
        self.norm = LayerNorm(dim, eps=1e-6)
        self.pwconv1 = nn.Linear(dim, 4 * dim)
        self.act = nn.GELU()
        self.pwconv2 = nn.Linear(4 * dim, dim)
        self.gamma = (nn.Parameter(layer_scale_init_value * torch.ones((dim)), requires_grad=True)
                      if layer_scale_init_value > 0 else None)
        self.drop_path = nn.Identity()

    def forward(self, x):
        raise RuntimeError("Block is fused into the libacx kernels; call the ConvNeXt forward methods")


class _STFT(nn.Module):
    """Holds the frozen windowed-DFT conv kernels under the torchlibrosa key names."""

    def __init__(self, n_fft, hop_length):
        super().__init__()
        self.n_fft, self.hop_length = n_fft, hop_length
        n_out = n_fft // 2 + 1
        self.conv_real = nn.Conv1d(1, n_out, kernel_size=n_fft, stride=hop_length, bias=False)
        self.conv_imag = nn.Conv1d(1, n_out, kernel_size=n_fft, stride=hop_length, bias=False)
        real, imag = windowed_dft(n_fft)
        self.conv_real.weight.data = real
        self.conv_imag.weight.data = imag
        for p in self.parameters():
            p.requires_grad = False


class Spectrogram(nn.Module):
    def __init__(self, n_fft=1024, hop_length=320, **_unused):
        super().__init__()
        self.stft = _STFT(n_fft, hop_length)


class LogmelFilterBank(nn.Module):
    def __init__(self, sr=32000, n_fft=1024, n_mels=224, fmin=50, fmax=14000, **_unused):
        super().__init__()
        self.melW = nn.Parameter(slaney_mel_filterbank(sr, n_fft, n_mels, fmin, fmax), requires_grad=False)


class ConvNeXt(nn.Module):
    r"""ConvNeXt audio tagger, B200-native.  Constructor signature follows CX:145-158."""

    def __init__(self, in_chans=3, num_classes=1000, depths=[3, 3, 9, 3], dims=[96, 192, 384, 768],
                 drop_path_rate=0.0, use_pydub_augment=False, use_roll_augment=False, use_speed_perturb=False,
                 use_torchaudio=False, layer_scale_init_value=1e-6, head_init_scale=1.0):
        super().__init__()
        if list(depths) != list(DEPTHS) or list(dims) != list(DIMS):
            raise NotImplementedError("the B200 path implements ConvNeXt-Tiny (depths [3,3,9,3], dims [96,192,384,768])")
        if drop_path_rate != 0.0:
            raise NotImplementedError("drop_path_rate must be 0.0 (inference); pass drop_path_rate=0.0 as "
                                      "ConvNeXt.from_pretrained does (CX:499-505)")
        if use_torchaudio or use_pydub_augment or use_roll_augment or use_speed_perturb:
            raise NotImplementedError("training-time augmentations / the torchaudio front end are out of scope")
        if layer_scale_init_value <= 0:
            raise NotImplementedError("layer scale (gamma) is required")
        self.use_torchaudio = False
        self.use_pydub_augment = self.use_roll_augment = self.use_speed_perturb = False
        # hard-coded by the reference ctor (CX:161-174)
        self.spectrogram_extractor = Spectrogram(n_fft=1024, hop_length=320)
        self.logmel_extractor = LogmelFilterBank(sr=32000, n_fft=1024, n_mels=224, fmin=50, fmax=14000)
        self.bn0 = nn.BatchNorm2d(224)
        self.downsample_layers = nn.ModuleList()
        stem = nn.Sequential(nn.Conv2d(3, dims[0], kernel_size=(4, 4), stride=(4, 4)),
                             LayerNorm(dims[0], eps=1e-6, data_format="channels_first"))
        self.downsample_layers.append(stem)
        for i in range(3):
            self.downsample_layers.append(nn.Sequential(
                LayerNorm(dims[i], eps=1e-6, data_format="channels_first"),
                nn.Conv2d(dims[i], dims[i + 1], kernel_size=2, stride=2)))
        self.stages = nn.ModuleList()
        for i in range(4):
            self.stages.append(nn.Sequential(*[
                Block(dim=dims[i], drop_path=0.0, layer_scale_init_value=layer_scale_init_value)
                for _ in range(depths[i])]))
        self.norm = nn.LayerNorm(dims[-1], eps=1e-6)
        self.head_audioset = nn.Linear(dims[-1], num_classes)
        self.apply(self._init_weights)
        self.head_audioset.weight.data.mul_(head_init_scale)
        self.head_audioset.bias.data.mul_(head_init_scale)
        self._engine = None
        self._engine_key = None
        self.precision = os.environ.get("ACX_PRECISION", "bf16")

    def _init_weights(self, m):
        if isinstance(m, (nn.Conv2d, nn.Linear)):                  # CX:263-267
            nn.init.trunc_normal_(m.weight, std=0.02, a=-2.0, b=2.0)
            nn.init.constant_(m.bias, 0)

    # ---- engine cache ------------------------------------------------------------------------------
    def set_precision(self, precision):
        """"bf16" (tensor-core path, default) or "fp32" (fp32-accurate SIMT path)."""
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        self.precision = precision
        self._engine = None
        return self

    def refresh_packed_weights(self):
        """Drop the repacked weights (call after mutating parameters in place)."""
        self._engine = None

    def _apply(self, fn, *a, **k):
        self._engine = None
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, *a, **k):
        self._engine = None
        return super().load_state_dict(*a, **k)

    def _get_engine(self):
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            raise _native.NativeError(
                "audioset-convnext-inf_b200 runs on a B200 GPU only: move the model to CUDA (there is no CPU path)")
        if self.head_audioset.out_features != 527 or self.downsample_layers[0][0].weight.shape != (96, 1, 4, 4):
            raise NotImplementedError("only the audio-tagging configuration built by convnext_tiny(after_stem_dim="
                                      "[252, 56]) is implemented (527 classes, 1-channel 4x4/s4 stem)")
        key = (str(dev), self.precision)
        if self._engine is None or self._engine_key != key:
            self._engine = Engine(self.state_dict(), dev, self.precision)
            self._engine_key = key
        return self._engine

    def _check_inference(self, mixup_lambda):
        if self.training:
            raise RuntimeError("inference only: call model.eval() first (the reference's training-mode branches -- "
                               "augmentation, SpecAugment, mixup, BatchNorm updates -- are out of scope)")
        if mixup_lambda is not None:
            raise NotImplementedError("mixup is training-only")

    def _prep(self, x, mixup_lambda):
        self._check_inference(mixup_lambda)
        if x.dim() != 2:
            raise ValueError(f"expected a (batch, samples) waveform, got shape {tuple(x.shape)}")
        eng = self._get_engine()
        x = x.detach().to(device=eng.device, dtype=torch.float32).contiguous()
        self._check_amplitude(eng, x)
        return eng, x

    @staticmethod
    def _check_amplitude(eng, x):
        if os.environ.get("ACX_CHECK_AMPLITUDE") == "1" and eng.precision == "bf16" and x.numel():
            # debugging aid (one reduction + sync per call): the bf16-mode front end carries samples as 2^8-scaled fp16
            # pairs, so |x| must stay below 255 (INTEGRATION.md, input contract); the fp32-accurate mode has no such bound
            amax = float(x.abs().amax())
            if not amax < 255.0:
                raise ValueError(f"waveform amplitude {amax:g} exceeds the bf16-mode front end's range (|x| < 255): "
                                 "normalise to [-1, 1] like torchaudio.load / int16 / 32767, or use set_precision('fp32')")

    # ---- the three inference entry points --------------------------------------------------------
    def forward(self, x, mixup_lambda=None):
        eng, x = self._prep(x, mixup_lambda)
        out = eng.run(x, want=("logits",))
        return {"clipwise_output": out["probs"], "clipwise_logits": out["logits"]}

    def forward_scene_embeddings(self, x, mixup_lambda=None):
        eng, x = self._prep(x, mixup_lambda)
        return eng.run(x, want=("scene",))["scene"]

    def forward_frame_embeddings(self, x, mixup_lambda=None):
        eng, x = self._prep(x, mixup_lambda)
        return eng.run(x, want=("frame",))["frame"]

    def forward_all(self, x, lengths=None):
        """One pass for everything (the reference demo runs three, demo_convnext.py:73-104).

        lengths: None, or one length per clip (a host sequence or CPU tensor of B ints, each in [7360, x.shape[1]]) for a
        RAGGED batch: clip b is x[b, :lengths[b]], and samples past it are never read.  Every output of clip b then equals
        forward_all(x[b:b + 1, :lengths[b]]) bit for bit; "frame_embeddings" is (B, 768, T', 7) with T' the canvas's frame
        count and zeros past each clip's own count, which "frame_lengths" ((B,) int64) gives.  A clip's result depends on
        its exact length (reflect padding at its end, frame count), so this is NOT what the reference computes for a
        zero-padded batch such as AudioCaps' BasicCollate output: forward(x_padded) still gives that."""
        eng, x = self._prep(x, None)
        out = eng.run(x, want=("logits", "scene", "frame"), lengths=lengths)
        res = {"clipwise_output": out["probs"], "clipwise_logits": out["logits"],
               "scene_embeddings": out["scene"], "frame_embeddings": out["frame"]}
        if lengths is not None:
            h3 = [out_time_dims(int(n))[1][3] for n in lengths]
            res["frame_lengths"] = torch.tensor(h3, dtype=torch.int64).to(x.device)
        return res

    def forward_windows(self, recordings, window_samples=320000, hop_samples=32000, frame_embeddings=False,
                        sample_rate=32000):
        """Tag long recordings window by window, each window as a clip of its own (the model's training condition).

        recordings: one 1-D tensor or a sequence of 1-D tensors of any lengths, on the host or the device; float32, int16
        PCM (converted x / 32767. in the prep kernel) or any other float dtype (converted to float32).  Windows of
        `window_samples` start every `hop_samples` samples; a recording whose windows do not end at its last sample gets
        one more, end-aligned window, and one shorter than a window gets one window at its own length
        (windows.plan_windows).  The windows are read in place from one buffer holding the recordings end to end (int16
        when every recording is int16, else float32), never copied out, and may overlap.

        Returns, on the model's device, one row per window in recording order, start ascending: "clipwise_output" and
        "clipwise_logits" (N, 527), "scene_embeddings" (N, 768), and (N,) int64 "recording", "start" and "length"; with
        frame_embeddings=True also "frame_embeddings" (N, 768, T', 7), T' the frame count of a full window, zero past each
        window's own count, which "frame_lengths" gives.  Row i equals
        forward_all(recordings[recording_i][start_i : start_i + length_i][None]) bit for bit, and a window never reads a
        sample outside itself.  Every argument is checked before anything is launched.

        sample_rate: the recordings' rate in Hz, a positive int or one per recording.  Recordings not at 32 kHz are first
        resampled on the GPU (preprocess.resample: torchaudio's filter, exact length ceil(32000 * n / rate)) into one
        float32 buffer, and the windows are planned on the resampled lengths: window_samples, hop_samples and the returned
        "start" / "length" are then in 32 kHz samples of the RESAMPLED recording (seconds = start / 32000), and row i
        equals forward_windows of the resampled recordings passed at 32 kHz, bit for bit.  A recording whose resampled
        length is under 7360 samples raises ValueError.  With every rate at 32 kHz (the default) nothing is resampled and
        int16 recordings stay int16."""
        self._check_inference(None)
        recs = preprocess.check_waveforms(recordings, "recording")
        rates = preprocess.sample_rates(sample_rate, len(recs))
        resample = any(r != preprocess.SAMPLE_RATE for r in rates)
        lengths = [preprocess.resampled_length(r.numel(), sr) for r, sr in zip(recs, rates)]
        plan = plan_windows(lengths, window_samples, hop_samples)
        eng = self._get_engine()
        dev = eng.device
        if resample:
            buf = preprocess.resample_packed(recs, rates, preprocess.SAMPLE_RATE, dev)[0]
            pcm = False
        else:
            buf = preprocess.pack_waveforms(recs, dev)
            pcm = buf.dtype == torch.int16
        if not pcm:
            self._check_amplitude(eng, buf)
        want = ("logits", "scene", "frame") if frame_embeddings else ("logits", "scene")
        out = eng.run_windows(buf, plan, want)
        res = {"clipwise_output": out["probs"], "clipwise_logits": out["logits"], "scene_embeddings": out["scene"],
               "recording": plan.recording.to(dev), "start": plan.start.to(dev), "length": plan.length.to(dev)}
        if frame_embeddings:
            res["frame_embeddings"] = out["frame"]
            h3 = [out_time_dims(n)[1][3] for n in plan.length.tolist()]
            res["frame_lengths"] = torch.tensor(h3, dtype=torch.int64).to(dev)
        return res

    def open_stream(self, n_streams=1, window_samples=320000, hop_samples=32000, sample_rate=32000,
                    frame_embeddings=False, piece_seconds=10, detection=None):
        """Tag `n_streams` live audio streams window by window as their samples arrive; returns a stream.StreamTagger.

        s.push(chunks) appends new samples: one 1-D tensor (n_streams == 1) or a sequence of n_streams entries, each a
        1-D tensor or array of any length (1 sample, or far more than a window) on the host or the device; float32, int16
        PCM (read x / 32767. with a correctly rounded division) or any other float dtype; None or empty for nothing new.
        s.close(streams=None) ends the given streams (an index, a sequence, or None for every open one).  Both return
        the rows of the windows that became complete during the call, in the dict forward_windows returns: rows
        stream-major with "start" ascending ("recording" is the stream index), possibly zero rows.  A regular window
        [k hop, k hop + window) comes back from the call in which its last sample arrives; close adds the end-aligned
        tail window and, for a stream shorter than a window, its one own-length window (windows.plan_windows' rules).

        For every stream i, its rows from all calls in order equal forward_windows(rec_i, window_samples, hop_samples,
        frame_embeddings=frame_embeddings, sample_rate=rate_i) bit for bit, however the stream was cut into chunks;
        rec_i is the stream's chunks concatenated (int16 chunks converted x / 32767 first).  sample_rate is an int or one
        per stream; a stream not at 32 kHz is resampled on the GPU as it arrives, and "start" / "length" are in 32 kHz
        samples of the resampled stream.

        Device memory is allocated here and does not grow: one float32 ring per stream (window + one piece of samples,
        plus a window-long mirror) and, for streams not at 32 kHz, an input ring of one piece plus the filter's taps.
        A push longer than `piece_seconds` of a stream's audio is appended and tagged piece by piece within the call.
        Work runs on the current CUDA stream.  A wrong chunk count, a chunk that is not 1-D or has a bad dtype, a push
        to a closed stream, a bad rate, or a stream under 7360 samples (after resampling) at close raises ValueError
        before anything is copied or launched, and leaves every stream unchanged.

        detection: None, or a sed.Detection.  With one, every push / close result also has "activity" (the activity bins
        that became final during the call) and "events" (the events that became final), keyed as sed.detect returns
        them, "recording" being the stream index.  For every stream, its activity rows from all calls equal the rows of
        sed.detect(forward_windows(whole stream, sample_rate=rate), detection)["activity"], and its events from all calls,
        stably sorted by (class, onset), equal that recording's events, bit for bit.  It needs hop_samples <=
        window_samples and adds a fixed row ring and event state per stream (s.detection_bytes; stream.BinPlanner);
        each call with new bins reads one event count back from the device per piece.  None changes nothing."""
        from .stream import StreamTagger
        return StreamTagger(self, n_streams, window_samples, hop_samples, sample_rate, frame_embeddings, piece_seconds,
                            detection)

    def forward_logmel(self, x):
        """Normalised log-mel (B, T, 224): the tensor the reference has after bn0 (CX:298-306)."""
        eng, x = self._prep(x, None)
        return eng.run(x, want=("logmel",))["logmel"]

    # ---- checkpoints -------------------------------------------------------------------------------
    @classmethod
    def from_pretrained(cls, pretrained_checkpoint_path, map_location=None, use_auth_token=None):
        """CX:404-511: local file, Zenodo URL or Hugging Face id -> convnext_tiny([252,56]) with the
        checkpoint loaded.  Returns the model in training mode like the reference (call .eval())."""
        if os.path.isfile(pretrained_checkpoint_path):
            path_ = pretrained_checkpoint_path
        elif "https" in pretrained_checkpoint_path:
            dpath_ = os.path.join(torch.hub.get_dir(), "checkpoints")
            os.makedirs(dpath_, exist_ok=True)
            fname = os.path.basename(pretrained_checkpoint_path).replace("?download=1", "")
            path_ = os.path.join(dpath_, fname)
            torch.hub.download_url_to_file(pretrained_checkpoint_path, path_)
        else:
            from huggingface_hub import hf_hub_download
            from huggingface_hub.utils import RepositoryNotFoundError
            model_id, _, revision = pretrained_checkpoint_path.partition("@")
            try:
                path_ = hf_hub_download(model_id, HF_PYTORCH_WEIGHTS_NAME, repo_type="model",
                                        revision=revision or None, library_name="audioset-convnext",
                                        token=use_auth_token)
            except RepositoryNotFoundError:
                print(f"Could not download '{model_id}' model (private, gated or missing repository).")
                return None
            try:
                hf_hub_download(model_id, HF_CONFIG_NAME, repo_type="model", revision=revision or None,
                                library_name="audioset-convnext", token=use_auth_token)
            except Exception:  # noqa: BLE001 -- best effort, as in the reference (CX:474-493)
                pass
        model = convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56],
                              use_speed_perturb=False)
        load_checkpoint(model, path_, map_location or "cpu")
        return model


def load_checkpoint(model, path, map_location="cpu"):
    """`.safetensors` strict load (CX:507) or a torch `.pth` holding {"model": state_dict}
    (evaluate_convnext_on_audioset.py:36-38)."""
    # Decided by what the file IS, not by its first bytes looking like something: a safetensors file starts with a
    # little-endian u64 header length whose low bytes can be anything (0x80.., "PK"), so the extension wins, then a
    # real zip check, then a parse of the safetensors header; only what is left goes to torch.load.
    import zipfile
    ext = os.path.splitext(str(path))[1].lower()
    is_torch = ext in (".pth", ".pt", ".ckpt", ".bin")
    if not is_torch and ext != ".safetensors":
        is_torch = zipfile.is_zipfile(path) or not _looks_like_safetensors(path)
    if is_torch:
        ckpt = torch.load(path, map_location=map_location, weights_only=True)
        model.load_state_dict(ckpt["model"] if "model" in ckpt else ckpt)
    else:
        from safetensors.torch import load_model as st_load_model
        st_load_model(model, path)
        model._engine = None
    return model


def _looks_like_safetensors(path):
    import json
    import struct
    try:
        size = os.path.getsize(path)
        with open(path, "rb") as fh:
            (n,) = struct.unpack("<Q", fh.read(8))
            if n <= 0 or n > size - 8 or n > (100 << 20):
                return False
            return isinstance(json.loads(fh.read(n)), dict)
    except Exception:  # noqa: BLE001 -- anything unparsable is not safetensors
        return False


def convnext_tiny(pretrained=False, strict=False, in_22k=False, drop_path_rate=0.1, after_stem_dim=[56],
                  use_speed_perturb=False, use_pydub_augment=False, use_roll_augment=False, **kwargs):
    """Factory with the reference signature (CX:641-651).  Only the configuration every reference
    caller uses is implemented: after_stem_dim=[252, 56], drop_path_rate=0.0, pretrained=False."""
    if pretrained:
        raise NotImplementedError("ImageNet-pretrained initialisation needs network access; load an AudioSet "
                                  "checkpoint with ConvNeXt.from_pretrained instead")
    after_stem_dim = list(after_stem_dim)
    if after_stem_dim != [252, 56]:
        if after_stem_dim in ([56], [112], [504, 28], [504, 56]):
            raise NotImplementedError(f"after_stem_dim={after_stem_dim}: only the [252, 56] stem (4x4, stride 4, "
                                      "pad (4,0)) used by the released checkpoint is implemented")
        raise ValueError("ERROR: after_stem_dim can be set to 56 or 112 or [252,56]")   # CX:701-703
    model = ConvNeXt(in_chans=1, num_classes=527, depths=[3, 3, 9, 3], dims=[96, 192, 384, 768],
                     drop_path_rate=drop_path_rate, use_speed_perturb=use_speed_perturb,
                     use_pydub_augment=use_pydub_augment, use_roll_augment=use_roll_augment, **kwargs)
    stem_audioset = nn.Conv2d(1, 96, kernel_size=(4, 4), stride=(4, 4), padding=(4, 0))   # CX:688-691
    nn.init.trunc_normal_(stem_audioset.weight, std=0.02, a=-2.0, b=2.0)
    nn.init.constant_(stem_audioset.bias, 0)
    model.downsample_layers[0][0] = stem_audioset
    return model
