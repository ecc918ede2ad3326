"""CPU: host side of resampling at any sample rate -- the exact output length, the segment table and its tiles, rate
validation, the short-after-resampling checks of forward_windows / extract_clipwise, and the argument checks of the
acx_resample_segments entry points (all return before touching a device)."""
import math

import numpy as np
import pytest
import torch

import audioset_convnext_inf_b200 as acx
from audioset_convnext_inf_b200 import _native
from audioset_convnext_inf_b200.engine import MIN_RAGGED_LEN
from audioset_convnext_inf_b200.preprocess import (resampled_length, sample_rates, segment_tiles, segment_tiling,
                                                   sinc_resample_taps)

RATES = (44100, 22050, 48000, 96000, 16000, 8000, 11025, 88200, 24000, 192000)


def test_exact_length_is_the_integer_ceil():
    for rate in RATES:
        g = math.gcd(rate, 32000)
        for n in (0, 1, 2, 7, 441, 90569, 10 ** 6 + 3):
            assert resampled_length(n, rate) == -(-(32000 // g) * n // (rate // g)), (rate, n)
    assert resampled_length(90569, 44100) == 65720
    assert resampled_length(12345, 32000) == 12345                      # same rate: unchanged
    assert resampled_length(4_147_200_000, 48000) == 2_764_800_000      # a day at 48 kHz, past 2^31 on both sides
    n = 2 ** 31 + 7
    assert resampled_length(n, 44100) == -(-320 * n // 441)


def test_torchaudio_drops_a_sample_where_the_exact_length_does_not():
    TAF = pytest.importorskip("torchaudio.functional")
    n = 90569
    got = TAF.resample(torch.zeros(1, n), 44100, 32000).shape[-1]
    assert got == 65719 and resampled_length(n, 44100) == 65720
    for m in (1000, 44100, 90568):                                      # below it both agree
        assert TAF.resample(torch.zeros(1, m), 44100, 32000).shape[-1] == resampled_length(m, 44100)


def test_tiling_of_common_rates():
    for rate in RATES:
        taps, width, orig, new = sinc_resample_taps(rate, 32000)
        frames, groups = segment_tiling(orig, new, width)
        assert frames % 32 == 0 and 32 <= frames <= 256
        phases = 256 // frames * 4                                      # phase warps x 4 phases per thread
        assert groups == -(-new // phases), rate
        assert groups * phases >= new
    assert segment_tiling(441, 320, 9) == (32, 10)                      # 44.1 kHz: 32 frames x 32 phases per tile
    assert segment_tiling(3, 2, 10) == (256, 1)                         # 48 kHz: 256 frames x 4 phases (2 used)


def test_tiling_refuses_a_tile_that_does_not_fit():
    _, width, orig, new = sinc_resample_taps(44056, 32000)             # 5507 / 4000: a 5525-tap filter
    with pytest.raises(ValueError, match="shared memory"):
        segment_tiling(orig, new, width)


def test_segment_tiles_prefix():
    start, total = segment_tiles([65720, 1, 0, 320 * 32, 320 * 32 + 1], 32, 10, 320)
    # frames: 206, 1, 0, 32, 33 -> frame tiles 7, 1, 0, 1, 2 -> x 10 phase groups
    assert start.dtype == torch.int64 and start.tolist() == [0, 70, 80, 80, 90]
    assert total == 110
    start, total = segment_tiles([2_764_800_000], 256, 1, 2)           # one segment past 2^31 outputs
    assert start.tolist() == [0] and total == -(-(2_764_800_000 // 2) // 256)
    start, total = segment_tiles([], 32, 10, 320)
    assert start.numel() == 0 and total == 0


def test_sample_rate_validation():
    assert sample_rates(44100, 3) == [44100] * 3
    assert sample_rates(np.int64(48000), 1) == [48000]
    assert sample_rates([44100, 32000], 2) == [44100, 32000]
    for bad in (0, -44100, 44100.0, "44100", True, None, [44100], [44100, 0], [44100, 4.41e4], (44100, None)):
        with pytest.raises(ValueError, match="sample_rate"):
            sample_rates(bad, 2)


def test_resample_argument_checks_before_any_device_work():
    with pytest.raises(ValueError, match="1-D"):
        acx.preprocess.resample(torch.zeros(2, 100), 44100)
    with pytest.raises(ValueError, match="dtype"):
        acx.preprocess.resample(torch.zeros(100, dtype=torch.int32), 44100)
    with pytest.raises(ValueError, match="sample_rate"):
        acx.preprocess.resample([torch.zeros(100)] * 2, [44100])
    with pytest.raises(ValueError, match="new_freq"):
        acx.preprocess.resample(torch.zeros(100), 44100, new_freq=0)


class _CpuModel(torch.nn.Module):
    """Stands in for a model: the checks below must raise before anything reaches a device."""

    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.zeros(1))


def test_forward_windows_validates_rates_and_resampled_lengths_first():
    m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56]).eval()
    short = torch.zeros(resampled_length_inverse(MIN_RAGGED_LEN - 1, 44100))
    assert resampled_length(short.numel(), 44100) == MIN_RAGGED_LEN - 1
    with pytest.raises(ValueError, match="recording 1 has 7359 samples"):
        m.forward_windows([torch.zeros(500000), short], sample_rate=44100)
    with pytest.raises(ValueError, match="sample_rate has 1 entries"):
        m.forward_windows([torch.zeros(500000), torch.zeros(500000)], sample_rate=[44100])
    with pytest.raises(ValueError, match="sample_rate"):
        m.forward_windows(torch.zeros(500000), sample_rate=44100.5)
    with pytest.raises(ValueError, match="sample_rate"):
        m.forward_windows(torch.zeros(500000), sample_rate=0)
    # 7360 samples at 8 kHz are 29440 at 32 kHz: long enough once resampled, too short to be passed as 32 kHz
    with pytest.raises(ValueError, match="recording 0 has 7000 samples"):
        m.forward_windows(torch.zeros(7000))
    with pytest.raises(_native.NativeError):                             # passes every check, then needs the GPU
        m.forward_windows(torch.zeros(7000), sample_rate=8000)


def test_extract_clipwise_validates_rates_and_resampled_lengths_first():
    m = _CpuModel()
    clips = [np.zeros(50000, np.float32), np.zeros(resampled_length_inverse(MIN_RAGGED_LEN - 1, 48000), np.float32)]
    with pytest.raises(ValueError, match="clip 1 has 7359 samples"):
        acx.extract.extract_clipwise(m, clips, sample_rate=48000)
    with pytest.raises(ValueError, match="sample_rate has 3 entries"):
        acx.extract.extract_clipwise(m, clips, sample_rate=[48000] * 3)
    with pytest.raises(ValueError, match="sample_rate"):
        acx.extract.extract_clipwise(m, clips, sample_rate=-1)


def resampled_length_inverse(n_out, rate):
    """The longest input whose resampled length is n_out."""
    n = n_out * rate // 32000 + 2
    while resampled_length(n, rate) > n_out:
        n -= 1
    return n


# ---- C ABI: every resample_segments entry point checks its arguments before it touches a device -------------------------
_P = 4096        # a non-null dummy address: the calls below must fail before dereferencing anything


def _args(x=_P, x_len=10 ** 6, seg=_P, S=2, tiles=_P, n_tiles=100, taps=_P, orig=441, new=320, width=9, out=_P,
          out_len=10 ** 6):
    return (x, x_len, seg, S, tiles, n_tiles, taps, orig, new, width, out, out_len, 0)


@pytest.mark.parametrize("name", ["acx_resample_segments", "acx_resample_segments_pcm16"])
def test_segments_entry_points_reject_bad_arguments(name):
    fn = getattr(_native.load(), name)
    assert len(_native.SIGNATURES[name]) == len(_args())
    for kw in (dict(x=0), dict(seg=0), dict(tiles=0), dict(taps=0), dict(out=0)):
        assert fn(*_args(**kw)) == _native.ACX_ERR_ARG and "null" in _native.last_error(), kw
    for kw, msg in ((dict(S=0), "S=0"), (dict(S=-1), "S=-1"), (dict(x_len=0), "x_len=0"), (dict(x_len=-5), "x_len=-5"),
                    (dict(out_len=0), "out_len=0"), (dict(n_tiles=0), "n_tiles=0"), (dict(n_tiles=2 ** 31), "n_tiles"),
                    (dict(orig=0), "rates"), (dict(new=-320), "rates"), (dict(width=0), "width 0")):
        assert fn(*_args(**kw)) == _native.ACX_ERR_ARG and msg in _native.last_error(), kw
    assert fn(*_args(x_len=2 ** 40, S=0)) == _native.ACX_ERR_ARG and "x_len=1099511627776" in _native.last_error()
    assert fn(*_args(orig=5507, new=4000, width=9)) == _native.ACX_ERR_UNSUPPORTED
    assert fn(*([0] * len(_args()))) == _native.ACX_ERR_ARG                                       # everything null


def test_tiling_entry_point_rejects_bad_arguments():
    import ctypes
    lib = _native.load()
    a, b = ctypes.c_int(0), ctypes.c_int(0)
    assert lib.acx_resample_segments_tiling(441, 320, 9, None, ctypes.byref(b)) == _native.ACX_ERR_ARG
    assert lib.acx_resample_segments_tiling(441, 320, 9, ctypes.byref(a), None) == _native.ACX_ERR_ARG
    for o, n, w in ((0, 320, 9), (441, 0, 9), (441, 320, 0), (-1, 2, 3)):
        assert lib.acx_resample_segments_tiling(o, n, w, ctypes.byref(a), ctypes.byref(b)) == _native.ACX_ERR_ARG
    assert a.value == 0 and b.value == 0
