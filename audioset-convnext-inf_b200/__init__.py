"""audioset-convnext-inf_b200: B200-native (sm_100a) inference hot path of topel/audioset-convnext-inf.

    from audioset_convnext_inf_b200 import ConvNeXt, convnext_tiny
    model = ConvNeXt.from_pretrained("model.safetensors").cuda().eval()
    probs = model(waveform)["clipwise_output"]
"""
from . import _native  # noqa: F401
from .convnext import (Block, ConvNeXt, LayerNorm, LogmelFilterBank, Spectrogram, convnext_tiny,  # noqa: F401
                       load_checkpoint)
from .engine import Engine, PackedWeights, out_time_dims  # noqa: F401
from .pipeline import HostPipeline  # noqa: F401
from . import evalloop  # noqa: F401
from . import extract, preprocess, search, sed, stream, windows  # noqa: F401

__all__ = ["ConvNeXt", "convnext_tiny", "Block", "LayerNorm", "Engine", "HostPipeline", "load_checkpoint"]
