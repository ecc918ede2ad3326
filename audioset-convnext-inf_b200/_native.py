"""ctypes binding of libacx.so (C ABI in include/acx.h).  There is NO fallback: if the shared
library cannot be loaded (or built, when nvcc is present) every entry point raises."""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libacx.so")
_lock = threading.Lock()
_lib = None

ACX_BF16, ACX_F32 = 0, 1
ACX_ERR_ARG, ACX_ERR_UNSUPPORTED = 1, 3
EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_SCALE_RESID = 0, 1, 2

_vp, _i, _ll = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong

# name -> argtypes; every function returns int except the two noted below.
SIGNATURES = {
    "acx_version": [],
    "acx_last_error": [],
    "acx_device_ok": [],
    "acx_wave_prep": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "acx_wave_prep_pcm16": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "acx_power_mel_log": [_vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp],
    "acx_frontend_fused": [_vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "acx_frame_fold": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "acx_frame_fold_pcm16": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "acx_frontend_folded": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "acx_stem": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "acx_stem_gp": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp],
    "acx_dwconv_ln": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "acx_dwconv_tc": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "acx_layernorm_rows": [_vp, _vp, _vp, _vp, _ll, _i, _vp],
    "acx_dwconv_tc_gp": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "acx_gp_transpose": [_vp, _vp, _ll, _i, _i, _vp],
    "acx_gp_row_stats": [_vp, _vp, _ll, _i, _vp],
    "acx_ln_patchify_gp": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "acx_ln_patchify": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "acx_downsample_fused_gp": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "acx_gemm_bf16": [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp],
    "acx_gemm_bf16_gp_out": [_vp, _vp, _vp, _i, _i, _i, _vp, _vp],
    "acx_gemm_bf16_pw1_gp": [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp],
    "acx_gemm_bf16_pw2_gp": [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp],
    "acx_gemm_f32": [_vp, _ll, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp],
    "acx_mlp_fused": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp],
    "acx_mlp_fused_ln": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp],
    "acx_mlp_fused_gp": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp],
    "acx_head": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "acx_nhwc_to_nchw_f32": [_vp, _vp, _i, _i, _i, _i, _i, _vp],
    "acx_resample_fit": [_vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp],
    # ragged batches: the entry point above plus the device array of per-clip bounds (and, for the prep kernels, the
    # input row pitch), just before the stream
    "acx_wave_prep_ragged": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp],
    "acx_frame_fold_ragged": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp],
    "acx_stem_ragged": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp],
    "acx_stem_gp_ragged": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp],
    "acx_dwconv_tc_ragged": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp],
    "acx_dwconv_tc_gp_ragged": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp],
    "acx_dwconv_ln_ragged": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp],
    "acx_head_ragged": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp],
    "acx_nhwc_to_nchw_f32_ragged": [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp],
    # windows of one long recording: recording, its length, the (B,) int64 window offsets and the optional ragged lengths
    # first, then the arguments of the dense prep entry point
    "acx_wave_prep_windows": [_vp, _ll, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "acx_wave_prep_pcm16_windows": [_vp, _ll, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "acx_frame_fold_windows": [_vp, _ll, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "acx_frame_fold_pcm16_windows": [_vp, _ll, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    # any sample rate: segments packed in one buffer, (S, 4) int64 table and per-segment first tiles on the device
    "acx_resample_segments_tiling": [_i, _i, _i, _vp, _vp],
    "acx_resample_segments": [_vp, _ll, _vp, _i, _vp, _ll, _vp, _i, _i, _i, _vp, _ll, _vp],
    "acx_resample_segments_pcm16": [_vp, _ll, _vp, _i, _vp, _ll, _vp, _i, _i, _i, _vp, _ll, _vp],
    # live streams: packed chunks scattered into per-stream rings ((S, 6) int64 table), and the resampler reading and
    # writing rings ((S, 8) int64 table; otherwise the arguments of acx_resample_segments)
    "acx_stream_append": [_vp, _ll, _vp, _i, _vp, _ll, _vp],
    "acx_stream_append_pcm16": [_vp, _ll, _vp, _i, _vp, _ll, _vp],
    "acx_resample_stream": [_vp, _ll, _vp, _i, _vp, _ll, _vp, _i, _i, _i, _vp, _ll, _vp],
    # sound event detection: bins averaged from (M, 4) int64 row ranges; events from (S, 6) int64 sequences, in a count
    # phase (0) and a write phase (1)
    "acx_window_activity": [_vp, _ll, _vp, _ll, _vp, _vp],
    "acx_detect_events": [_vp, _ll, _vp, _i, _vp, _vp, _ll, _ll, _ll, _vp, _vp, _vp, _i, _vp, _vp, _ll, _vp],
    # query by example: fp64 row norms, the (Q, N) fp32 cosine score block, and the per-query top k over it (optional
    # (N, 2) int64 neighbour ranges, caller-owned workspace sized by the host query)
    "acx_row_norms": [_vp, _ll, _i, _vp, _vp],
    "acx_cosine_scores": [_vp, _vp, _ll, _vp, _vp, _ll, _i, _vp, _vp],
    "acx_search_topk_workspace": [_ll, _ll, _vp],
    "acx_search_topk": [_vp, _ll, _ll, _vp, _i, _vp, _vp, _vp, _vp],
    # tagging metrics: per-class (P, U2, S_lo, S_hi) counts of classes [c0, c0 + kc) of (N, K) scores and uint8 targets,
    # caller-owned workspace sized by the host query
    "acx_tagging_metrics_workspace": [_ll, _i, _vp],
    "acx_tagging_metrics": [_vp, _ll, _i, _i, _i, _vp, _vp, _vp, _vp],
}


class NativeError(RuntimeError):
    pass


def lib_path():
    return _LIB_PATH


def load():
    """Load (building first if the .so is absent and nvcc exists).  Raises NativeError."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.isfile(_LIB_PATH):
            try:
                from . import build as _build
                _build.build()
            except Exception as e:  # noqa: BLE001
                raise NativeError(
                    f"libacx.so is missing at {_LIB_PATH} and could not be built ({e}). "
                    "The B200 path has no CPU or PyTorch fallback.") from e
        try:
            lib = ctypes.CDLL(_LIB_PATH)
        except OSError as e:
            raise NativeError(f"cannot load {_LIB_PATH}: {e}") from e
        for name, argtypes in SIGNATURES.items():
            try:
                fn = getattr(lib, name)
            except AttributeError as e:
                raise NativeError(f"{_LIB_PATH} does not export {name}; rebuild it") from e
            fn.argtypes = argtypes
            fn.restype = ctypes.c_char_p if name == "acx_last_error" else ctypes.c_int
        _lib = lib
    return _lib


def last_error():
    msg = load().acx_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc, what):
    if rc != 0:
        raise NativeError(f"{what} failed (code {rc}): {last_error()}")


def call(name, *args):
    """Invoke an int-returning entry point and raise on a non-zero code."""
    check(getattr(load(), name)(*args), name)
