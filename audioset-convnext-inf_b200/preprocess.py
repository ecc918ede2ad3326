"""Clip preparation in front of the hot path (SURVEY §8 row f4): what reference demo_convnext.py:52-67 does with
torchaudio on the host -- resample to 32 kHz, then constant-pad or crop to 10 s -- as ONE libacx launch on the GPU.

The resampler is torchaudio.functional.resample's algorithm (sinc interpolation, Hann-windowed, lowpass_filter_width 6,
rolloff 0.99), restated here: torchaudio is not a dependency of the product; tests/ compare against it.
"""
import ctypes
import math
import numbers

import numpy as np
import torch

from . import _native
from ._native import ACX_ERR_UNSUPPORTED

SAMPLE_RATE = 32000
CLIP_SAMPLES = 10 * SAMPLE_RATE        # demo_convnext.py:47-48


def _rate_params(orig_freq, new_freq, lowpass_filter_width=6, rolloff=0.99):
    """(orig, new, width): the rates divided by their gcd and the filter's half-width in input samples."""
    if int(orig_freq) != orig_freq or int(new_freq) != new_freq or orig_freq <= 0 or new_freq <= 0:
        raise ValueError("resample: frequencies must be positive integers")
    g = math.gcd(int(orig_freq), int(new_freq))
    orig, new = int(orig_freq) // g, int(new_freq) // g
    return orig, new, math.ceil(lowpass_filter_width * orig / (min(orig, new) * rolloff))


def sinc_resample_taps(orig_freq, new_freq, lowpass_filter_width=6, rolloff=0.99, dtype=torch.float32):
    """(taps (K, new) transposed polyphase kernel, width, orig, new) with orig/new reduced by their gcd.

    Same arithmetic, in the same order and dtype, as torchaudio's `_get_sinc_resample_kernel` when called from
    `resample(waveform_fp32, ...)` (it builds the kernel in the waveform's dtype): kernel[p, k] =
    sinc(pi t) * cos^2(pi t / (2 lw)) * scale with t = clamp((k - width)/orig - p/new) * base_freq, +-lw)."""
    orig, new, width = _rate_params(orig_freq, new_freq, lowpass_filter_width, rolloff)
    base_freq = min(orig, new) * rolloff
    idx = torch.arange(-width, width + orig, dtype=dtype)[None, None] / orig
    t = torch.arange(0, -new, -1, dtype=dtype)[:, None, None] / new + idx
    t *= base_freq
    t = t.clamp_(-lowpass_filter_width, lowpass_filter_width)
    window = torch.cos(t * math.pi / lowpass_filter_width / 2) ** 2
    t *= math.pi
    scale = base_freq / orig
    kernels = torch.where(t == 0, torch.tensor(1.0).to(t), t.sin() / t)
    kernels *= window * scale
    taps = kernels.to(torch.float32)[:, 0, :].t().contiguous()            # (K, new): lanes read consecutive phases
    return taps, width, orig, new


_TAPS_CACHE = {}


def _cached_taps(orig_freq, new_freq, device):
    key = (int(orig_freq), int(new_freq), device)
    if key not in _TAPS_CACHE:
        if int(orig_freq) == int(new_freq):
            # torchaudio's resample() returns the input unchanged: a 3-tap delta keeps the single launch (pad / crop)
            taps, width, orig, new = torch.tensor([[0.0], [1.0], [0.0]]), 1, 1, 1
        else:
            taps, width, orig, new = sinc_resample_taps(orig_freq, new_freq)
        _TAPS_CACHE[key] = (taps.to(device), width, orig, new)
    return _TAPS_CACHE[key]


def resample_fit(waveform, orig_freq, new_freq=SAMPLE_RATE, n_out=CLIP_SAMPLES):
    """waveform (B, L) or (L,) float32 CUDA tensor at orig_freq -> (B, n_out) at new_freq: resampled, then zero-padded
    or cropped to n_out samples (n_out=None keeps torchaudio's length ceil(new * L / orig)).  No CPU fallback."""
    if not waveform.is_cuda:
        raise RuntimeError("resample_fit needs a CUDA tensor: the B200 path has no CPU fallback")
    x = waveform.reshape(-1, waveform.shape[-1]).to(torch.float32).contiguous()
    B, L = x.shape
    taps, width, orig, new = _cached_taps(orig_freq, new_freq, x.device)
    target = -(-new * L // orig)
    n = target if n_out is None else int(n_out)
    out = torch.empty(B, n, device=x.device, dtype=torch.float32)
    _native.call("acx_resample_fit", x.data_ptr(), L, taps.data_ptr(), out.data_ptr(), n, B, L, orig, new, width, n,
                 torch.cuda.current_stream(x.device).cuda_stream)
    return out if waveform.dim() > 1 else out[0]


# ---- any sample rate: many waveforms of any lengths, one launch per distinct rate ----------------------------------------
def resampled_length(n, orig_freq, new_freq=SAMPLE_RATE):
    """Samples of an n-sample waveform at orig_freq once resampled to new_freq: ceil(new * n / orig) with the rates
    divided by their gcd, in exact integer arithmetic (n past 2^31 too); n when the rates are equal.  resample_fit(...,
    n_out=None) keeps the same length.  torchaudio computes it through a float32 tensor and can come out one sample short:
    for 44 100 -> 32 000 that first happens at n = 90 569 (torchaudio gives 65 719 samples, the exact ceil is 65 720)."""
    n = int(n)
    if int(orig_freq) == int(new_freq):
        return n
    orig, new, _ = _rate_params(orig_freq, new_freq)
    return -(-new * n // orig)


def sample_rates(sample_rate, count):
    """One rate per waveform: `sample_rate` is a positive int for all `count` waveforms, or a sequence of `count` positive
    ints.  Raises ValueError otherwise."""
    def ok(r):
        return isinstance(r, numbers.Integral) and not isinstance(r, bool) and int(r) > 0
    if ok(sample_rate):
        return [int(sample_rate)] * count
    if isinstance(sample_rate, (list, tuple)):
        if len(sample_rate) != count:
            raise ValueError(f"sample_rate has {len(sample_rate)} entries for {count} waveforms")
        for i, r in enumerate(sample_rate):
            if not ok(r):
                raise ValueError(f"sample_rate[{i}] = {r!r}: expected a positive int (samples per second)")
        return [int(r) for r in sample_rate]
    raise ValueError(f"sample_rate = {sample_rate!r}: expected a positive int or one positive int per waveform")


def segment_tiling(orig, new, width):
    """(tile_frames, phase_groups) of acx_resample_segments for reduced rates orig -> new: a host query, no launch.
    Raises ValueError for a rate pair whose tile does not fit in shared memory."""
    tf, pg = ctypes.c_int(0), ctypes.c_int(0)
    lib = _native.load()
    rc = lib.acx_resample_segments_tiling(orig, new, width, ctypes.byref(tf), ctypes.byref(pg))
    if rc == ACX_ERR_UNSUPPORTED:
        raise ValueError(f"resample: {_native.last_error()}")
    _native.check(rc, "acx_resample_segments_tiling")
    return tf.value, pg.value


def segment_tiles(out_lengths, tile_frames, phase_groups, new):
    """((S,) int64 first tile of each segment, total tiles): segment s owns ceil(ceil(n_s / new) / tile_frames) *
    phase_groups tiles, laid out one segment after another."""
    counts = [-(-(-(-int(n) // new)) // tile_frames) * phase_groups for n in out_lengths]
    start = np.zeros(len(counts), dtype=np.int64)
    if counts:
        start[1:] = np.cumsum(np.asarray(counts[:-1], dtype=np.int64))
    return torch.from_numpy(start), int(sum(counts))


def check_waveforms(waveforms, what="waveform"):
    """A list of 1-D tensors (host or device; a float dtype or int16 PCM) from one tensor or a sequence of array-likes."""
    if isinstance(waveforms, torch.Tensor):
        waveforms = [waveforms]
    ws = [w if isinstance(w, torch.Tensor) else torch.as_tensor(w) for w in waveforms]
    for i, w in enumerate(ws):
        if w.dim() != 1:
            raise ValueError(f"{what} {i} must be 1-D (samples), got shape {tuple(w.shape)}")
        if not (w.dtype == torch.int16 or w.is_floating_point()):
            raise ValueError(f"{what} {i} has dtype {w.dtype}: expected a float dtype or int16 PCM")
    return ws


def _pcm_to_float(src, dst):
    # the prep kernels' conversion, a correctly rounded fp32 division (not a reciprocal multiply)
    torch.div(src.to(dst.device).to(torch.float32), torch.tensor(32767.0, device=dst.device), out=dst)


def pack_waveforms(waveforms, device, pin_memory=False):
    """The waveforms end to end in one device buffer: int16 when every one is int16, else float32 (int16 converted by a
    correctly rounded x / 32767, other float dtypes cast).  A single contiguous float32 / int16 waveform already on the
    device is returned as it is, not copied.  pin_memory: a new host buffer is allocated in pinned memory."""
    w0 = waveforms[0] if len(waveforms) == 1 else None
    if w0 is not None and w0.device == device and w0.dtype in (torch.float32, torch.int16) and w0.is_contiguous():
        return w0.detach()
    pcm = bool(waveforms) and all(w.dtype == torch.int16 for w in waveforms)
    buf = torch.empty(sum(w.numel() for w in waveforms), dtype=torch.int16 if pcm else torch.float32, device=device,
                      pin_memory=pin_memory)
    base = 0
    for w in waveforms:
        dst = buf[base:base + w.numel()]
        if w.dtype == torch.int16 and not pcm:
            _pcm_to_float(w.detach(), dst)
        else:
            dst.copy_(w.detach())
        base += w.numel()
    return buf


def resample_packed(waveforms, rates, new_freq, device):
    """(out, lengths): checked 1-D waveforms at their `rates` resampled to new_freq into ONE float32 device buffer, end to
    end in input order; lengths[i] = resampled_length(len(waveforms[i]), rates[i], new_freq).  The inputs are packed by
    pack_waveforms; one acx_resample_segments(_pcm16) launch per distinct rate resamples all its waveforms, each exactly
    as acx_resample_fit of that waveform alone.  A waveform already at new_freq is copied unchanged (int16 converted
    x / 32767), as torchaudio's resample() returns it.  Every rate is checked before anything is copied or launched."""
    new_freq = int(new_freq)
    n_in = [w.numel() for w in waveforms]
    lengths = [resampled_length(n, r, new_freq) for n, r in zip(n_in, rates)]
    groups = {}
    for i, r in enumerate(rates):
        if r != new_freq and lengths[i] > 0:
            groups.setdefault(r, []).append(i)
    tilings = {}
    for r in groups:
        orig, new, width = _rate_params(r, new_freq)
        tilings[r] = segment_tiling(orig, new, width)
    x = pack_waveforms(waveforms, device)
    out = torch.empty(sum(lengths), dtype=torch.float32, device=device)
    in_off = np.concatenate([[0], np.cumsum(n_in, dtype=np.int64)]).tolist()
    out_off = np.concatenate([[0], np.cumsum(lengths, dtype=np.int64)]).tolist()
    for i, r in enumerate(rates):
        if r == new_freq and n_in[i]:
            src, dst = x[in_off[i]:in_off[i] + n_in[i]], out[out_off[i]:out_off[i] + lengths[i]]
            if src.dtype == torch.int16:
                _pcm_to_float(src, dst)
            else:
                dst.copy_(src)
    stream = torch.cuda.current_stream(device).cuda_stream
    entry = "acx_resample_segments_pcm16" if x.dtype == torch.int16 else "acx_resample_segments"
    for r, idx in groups.items():
        taps, width, orig, new = _cached_taps(r, new_freq, device)
        tile_frames, phase_groups = tilings[r]
        start, n_tiles = segment_tiles([lengths[i] for i in idx], tile_frames, phase_groups, new)
        seg = torch.tensor([[in_off[i], n_in[i], out_off[i], lengths[i]] for i in idx], dtype=torch.int64)
        table = torch.cat([seg.flatten(), start]).to(device)       # (S, 4) segments, then (S,) first tiles
        S = len(idx)
        _native.call(entry, x.data_ptr(), x.numel(), table.data_ptr(), S, table.data_ptr() + 8 * 4 * S, n_tiles,
                     taps.data_ptr(), orig, new, width, out.data_ptr(), out.numel(), stream)
    return out, lengths


def resample(waveforms, orig_freq, new_freq=SAMPLE_RATE, device=None):
    """Resample one 1-D waveform or a sequence of them to new_freq on the GPU.

    waveforms: 1-D tensors or array-likes of any lengths, on the host or the device; float32, int16 PCM (read as
    x / 32767 with a correctly rounded division) or any other float dtype (cast to float32).  orig_freq: a positive int,
    or one per waveform.  Returns a list of float32 tensors on `device` (default: the first CUDA waveform's device, else
    the current CUDA device), views of one packed buffer, in input order.

    The filter is torchaudio.functional.resample's (sinc_interp_hann, lowpass_filter_width 6, rolloff 0.99); each output
    equals resample_fit(waveform, orig_freq, new_freq, n_out=None) of that waveform alone, bit for bit, and has exactly
    resampled_length(len, orig_freq, new_freq) samples -- which torchaudio can undershoot by one (see there).  A waveform
    already at new_freq is returned unchanged (converted to float32), like torchaudio, without running a filter.  All
    waveforms at one rate are resampled by one launch."""
    ws = check_waveforms(waveforms)
    if not (isinstance(new_freq, numbers.Integral) and not isinstance(new_freq, bool) and new_freq > 0):
        raise ValueError(f"new_freq = {new_freq!r}: expected a positive int")
    rates = sample_rates(orig_freq, len(ws))
    if device is None:
        device = next((w.device for w in ws if w.is_cuda), None) or torch.device("cuda", torch.cuda.current_device())
    device = torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    if device.type != "cuda":
        raise RuntimeError("resample runs on the GPU: the B200 path has no CPU fallback")
    if not ws:
        return []
    out, lengths = resample_packed(ws, rates, new_freq, device)
    offs = np.concatenate([[0], np.cumsum(lengths, dtype=np.int64)]).tolist()
    return [out[offs[i]:offs[i + 1]] for i in range(len(ws))]


def tags_above(probs, threshold=0.25):
    """Indices of the classes whose probability exceeds `threshold`, per clip (demo_convnext.py:87-88)."""
    p = probs.detach()
    return [torch.nonzero(row > threshold).flatten().cpu().numpy() for row in p.reshape(-1, p.shape[-1])]
