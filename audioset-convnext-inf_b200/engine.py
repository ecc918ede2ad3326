"""Host-side orchestration of the hot path: weight repacking, workspace, kernel sequence.

Everything that touches numbers runs in libacx.so (hand-written sm_100a CUDA behind the C ABI in
include/acx.h); PyTorch only owns device memory and the stream.  Two arithmetic modes:

  "bf16"  activations / GEMM operands bf16, fp32 accumulation in TMEM (tcgen05), fp32 LayerNorm
          statistics; the front end runs split precision (x3: scaled fp16 pairs for the DFT, bf16 pairs for the mel
          product) so the log-mel keeps fp32-level accuracy.
  "fp32"  the fp32-accurate mode: same bandwidth kernels instantiated for float, SIMT fp32 GEMMs.

Kernel order per chunk of clips (reference convnext.py:287-331, forward_features :269-285):
  wave_prep -> front end -> stem -> [dwconv_ln -> pwconv1+GELU -> pwconv2+gamma+residual] x (3,3,9,3)
  with ln_patchify + GEMM between stages -> head (pool + LayerNorm + fc + sigmoid) / frame transpose.
"""
import collections
import os

import torch

from . import _native as N

DEPTHS = (3, 3, 9, 3)
DIMS = (96, 192, 384, 768)
N_FFT, HOP, N_MELS, N_BINS, N_CLASSES = 1024, 320, 224, 513, 527
BN0_EPS = 1e-5
FE_SCALE_LOG2 = 8          # == ACX_FE_SCALE_LOG2 in include/acx.h


def _p(t):
    return 0 if t is None else t.data_ptr()


class PackedWeights:
    """Kernel-friendly copies of the 190-entry state dict (SURVEY.md Appendix B).  Built once per
    (device, precision); the module drops it whenever parameters may have changed."""

    def __init__(self, sd, device, precision):
        assert precision in ("bf16", "fp32")
        self.precision = precision
        self.device = device
        adt = torch.bfloat16 if precision == "bf16" else torch.float32
        self.act_dtype = adt
        f32 = dict(device=device, dtype=torch.float32)

        def g(key):
            return sd[key].detach().to(**f32)

        # ---- front end -----------------------------------------------------------------------
        conv_real = g("spectrogram_extractor.stft.conv_real.weight")[:, 0, :]   # (513, 1024)
        conv_imag = g("spectrogram_extractor.stft.conv_imag.weight")[:, 0, :]
        melW = g("logmel_extractor.melW")                                         # (513, 224)
        assert conv_real.shape == (N_BINS, N_FFT) and melW.shape == (N_BINS, N_MELS), \
            "only the n_fft=1024 / 224-mel front end of convnext_tiny is supported"
        scale = g("bn0.weight") / torch.sqrt(g("bn0.running_var") + BN0_EPS)
        self.bn_scale = scale.contiguous()
        self.bn_shift = (g("bn0.bias") - g("bn0.running_mean") * scale).contiguous()
        # fp32-accurate path: dense windowed-DFT rows (re | im) and banded mel
        self.dft_f32 = torch.cat([conv_real, conv_imag], 0).contiguous()         # (1026, 1024)
        self.melT = melW.t().contiguous()                                          # (224, 513)
        nz = melW != 0
        idx = torch.arange(N_BINS, device=device)[:, None].expand(N_BINS, N_MELS)
        big = torch.full_like(idx, N_BINS)
        lo = torch.where(nz, idx, big).min(0).values
        hi = torch.where(nz, idx + 1, torch.zeros_like(idx)).max(0).values
        lo = torch.minimum(lo, hi)
        self.mel_lo = lo.to(torch.int32).contiguous()
        self.mel_hi = hi.to(torch.int32).contiguous()
        # tensor-core path: 64-bin chunks; only bins that feed a non-zero mel weight are computed
        used = nz.any(1).nonzero().flatten()
        k_end = int(used.max().item()) + 1 if used.numel() else 1
        self.n_chunks = (k_end + 63) // 64
        if precision == "bf16":
            nb = self.n_chunks * 64
            re = torch.zeros(nb, N_FFT, **f32)
            im = torch.zeros(nb, N_FFT, **f32)
            m = min(nb, N_BINS)
            re[:m], im[:m] = conv_real[:m], conv_imag[:m]
            dft = torch.stack([re.view(self.n_chunks, 64, N_FFT), im.view(self.n_chunks, 64, N_FFT)], 1)
            dft = dft.reshape(self.n_chunks * 128, N_FFT)
            self.dft_hi, self.dft_lo = _split_f16(dft * float(1 << FE_SCALE_LOG2))
            # folded form (frontend_folded.cu): None when the loaded rows do not have the real-input symmetry
            self.dftf = fold_dft_weights(conv_real, conv_imag, self.n_chunks)
            if self.dftf is not None:
                self.dftf_hi, self.dftf_lo = _split_f16(self.dftf * float(1 << FE_SCALE_LOG2))
            mw = torch.zeros(nb, 256, **f32)
            mw[:m, :N_MELS] = melW[:m]
            mel = mw.view(self.n_chunks, 64, 256).transpose(1, 2).reshape(self.n_chunks * 256, 64)
            self.melc_hi, self.melc_lo = _split_bf16(mel)

        # ---- stem ---------------------------------------------------------------------------
        self.stem_w = g("downsample_layers.0.0.weight").reshape(DIMS[0], 16).t().contiguous()  # (16, 96)
        self.stem_b = g("downsample_layers.0.0.bias").contiguous()
        self.stem_ln_w = g("downsample_layers.0.1.weight").contiguous()
        self.stem_ln_b = g("downsample_layers.0.1.bias").contiguous()

        # ---- downsample layers 1..3 ---------------------------------------------------------
        self.ds = []
        for i in range(1, 4):
            w = g(f"downsample_layers.{i}.1.weight")                 # (Cout, Cin, 2, 2)
            cout, cin = w.shape[0], w.shape[1]
            self.ds.append(dict(
                ln_w=g(f"downsample_layers.{i}.0.weight").contiguous(),
                ln_b=g(f"downsample_layers.{i}.0.bias").contiguous(),
                w=w.permute(0, 2, 3, 1).reshape(cout, 4 * cin).to(adt).contiguous(),   # k = (dy, dx, cin)
                b=g(f"downsample_layers.{i}.1.bias").contiguous()))
            if precision == "bf16":
                self.ds[-1]["w_fused"] = pack_downsample_weight(w).to(adt).contiguous()

        # ---- blocks -------------------------------------------------------------------------
        self.blocks = []
        for s in range(4):
            C = DIMS[s]
            stage = []
            for j in range(DEPTHS[s]):
                p = f"stages.{s}.{j}."
                stage.append(dict(
                    dw_w=g(p + "dwconv.weight").reshape(C, 49).t().to(adt).contiguous(),   # (49, C)
                    dw_b=g(p + "dwconv.bias").contiguous(),
                    ln_w=g(p + "norm.weight").contiguous(), ln_b=g(p + "norm.bias").contiguous(),
                    w1=g(p + "pwconv1.weight").to(adt).contiguous(), b1=g(p + "pwconv1.bias").contiguous(),
                    w2=g(p + "pwconv2.weight").to(adt).contiguous(), b2=g(p + "pwconv2.bias").contiguous(),
                    gamma=g(p + "gamma").contiguous()))
                if precision == "bf16" and s < 3:
                    stage[-1].update(fold_layernorm_into_pwconv1(g(p + "pwconv1.weight"), g(p + "pwconv1.bias"),
                                                                 g(p + "norm.weight"), g(p + "norm.bias")))
            self.blocks.append(stage)

        # ---- head ---------------------------------------------------------------------------
        self.norm_w, self.norm_b = g("norm.weight").contiguous(), g("norm.bias").contiguous()
        self.fc_w, self.fc_b = g("head_audioset.weight").contiguous(), g("head_audioset.bias").contiguous()


def fold_layernorm_into_pwconv1(w1, b1, ln_w, ln_b):
    """LayerNorm (CX:78) folded into pwconv1 (CX:79) for the tensor-core depthwise-conv path, whose output v is never
    normalised in memory:   pwconv1(LN(v)) = rstd * (v . W1'^T - mean * s) + b1'   with
        W1' = bf16(W1 * ln_w)   (the GEMM operand),   s_j = sum_c W1'[j, c]   (of the ROUNDED operand, so that the
        identity  sum_c (v_c - mean) W1'[j, c] = G_j - mean s_j  is exact),   b1' = b1 + W1 ln_b.
    The kernel computes (mean, rstd) per row from the same bf16 tile it multiplies."""
    w1f = (w1.double() * ln_w.double()[None, :]).to(torch.float32).to(torch.bfloat16).contiguous()
    return dict(w1f=w1f, s1=w1f.double().sum(1).to(torch.float32).contiguous(),
                b1f=(b1.double() + w1.double() @ ln_b.double()).to(torch.float32).contiguous())


def fold_dft_weights(conv_real, conv_imag, n_chunks, tol=1e-6):
    """Windowed-DFT rows (513, 1024) of the checkpoint -> the folded operand of acx_frontend_folded, or None.

    With E[0] = x[512], E[j] = x[j] + x[1024 - j], O[0] = 0, O[j] = x[j] - x[1024 - j] (acx_frame_fold) a frame's spectrum is
    re[k] = sum_j E[j] Wre'[k, j], im[k] = sum_j O[j] Wim'[k, j] IF the rows are even / odd about n = 512 and vanish at
    n = 0 -- which a periodic-Hann STFT matrix does (torchlibrosa Spectrogram, CX:179-187) but an arbitrary conv weight need
    not: the symmetry of the LOADED rows is checked (relative to the largest entry) and None returned otherwise, in which
    case the engine keeps the dense kernel.  Layout: per pair p of 64-bin chunks 256 rows x 512 --
    [re chunk 2p | re chunk 2p+1 | im chunk 2p | im chunk 2p+1], zero rows past the last used bin."""
    n_bins, n_fft = conv_real.shape
    h = n_fft // 2
    scale = max(conv_real.abs().max().item(), conv_imag.abs().max().item(), 1e-30)
    mir = torch.arange(n_fft - 1, h, -1, device=conv_real.device)            # 1023 .. 513 <-> j = 1 .. 511
    asym = max((conv_real[:, 1:h] - conv_real[:, mir]).abs().max().item(), (conv_imag[:, 1:h] + conv_imag[:, mir]).abs().max().item(),
               conv_real[:, 0].abs().max().item(), conv_imag[:, 0].abs().max().item(), conv_imag[:, h].abs().max().item())
    if asym > tol * scale:
        return None
    fre = torch.zeros(n_bins, h, device=conv_real.device, dtype=torch.float32)
    fim = torch.zeros_like(fre)
    fre[:, 0] = conv_real[:, h]
    fre[:, 1:] = 0.5 * (conv_real[:, 1:h] + conv_real[:, mir])
    fim[:, 1:] = 0.5 * (conv_imag[:, 1:h] - conv_imag[:, mir])
    n_pairs = (n_chunks + 1) // 2
    out = torch.zeros(n_pairs, 4, 64, h, device=conv_real.device, dtype=torch.float32)
    for c in range(n_chunks):
        lo, hi = 64 * c, min(64 * c + 64, n_bins)
        if hi > lo:
            out[c // 2, c % 2, : hi - lo] = fre[lo:hi]
            out[c // 2, 2 + c % 2, : hi - lo] = fim[lo:hi]
    return out.reshape(n_pairs * 256, h).contiguous()


def pack_downsample_weight(w):
    """Conv2d(k2, s2) weight (Cout, Cin, 2, 2) -> (Cout, 4 Cin) with k = ((dy * Cin/8 + g) * 2 + dx) * 8 + c8: the K order of
    acx_downsample_fused_gp, in which the two horizontally adjacent pixels of a patch are 32 contiguous bytes of a
    group-planar plane and of the operand row (CX:231-234)."""
    cout, cin = w.shape[0], w.shape[1]
    return w.reshape(cout, cin // 8, 8, 2, 2).permute(0, 3, 1, 4, 2).reshape(cout, 4 * cin)


def _split_f16(x):
    """fp16 hi + lo (22 mantissa bits) of an already-scaled fp32 tensor (include/acx.h, ACX_FE_SCALE_LOG2)."""
    hi = x.to(torch.float16)
    lo = (x - hi.to(torch.float32)).to(torch.float16)
    return hi.contiguous(), lo.contiguous()


def _split_bf16(x):
    hi = x.to(torch.bfloat16)
    lo = (x - hi.to(torch.float32)).to(torch.bfloat16)
    return hi.contiguous(), lo.contiguous()


def out_time_dims(L):
    """Frame count and per-stage heights for an L-sample clip (SURVEY.md section 0)."""
    T = L // HOP + 1
    H0 = (T + 4) // 4 + 1          # Conv2d(k=4, s=4, pad=(4,0)) over time
    hs = [H0, H0 // 2, (H0 // 2) // 2, ((H0 // 2) // 2) // 2]
    return T, hs


MIN_RAGGED_LEN = 7360      # shortest clip with h3 >= 1 (it also reflects: L > N_FFT / 2)


def check_lengths(lengths, B, L):
    """Per-clip lengths of a ragged batch -> list of B ints in [MIN_RAGGED_LEN, L]; ValueError otherwise."""
    if isinstance(lengths, torch.Tensor):
        if lengths.device.type != "cpu":
            raise ValueError("lengths must be a host sequence or a CPU tensor")
        lengths = lengths.tolist()
    try:
        ls = [int(n) for n in lengths]
    except (TypeError, ValueError) as e:
        raise ValueError(f"lengths must be a sequence of integers: {e}") from e
    if len(ls) != B:
        raise ValueError(f"lengths has {len(ls)} entries for a batch of {B} clips")
    bad = [n for n in ls if not MIN_RAGGED_LEN <= n <= L]
    if bad:
        raise ValueError(f"every length must lie in [{MIN_RAGGED_LEN}, {L}] (the canvas), got {bad[:4]}")
    return ls


def ragged_table(lengths):
    """(6, n) int32 table of a ragged chunk: per clip L, T, h0, h1, h2, h3 (the bound each kernel family reads)."""
    rows = []
    for n in lengths:
        T, hs = out_time_dims(n)
        rows.append([n, T] + hs)
    return torch.tensor(rows, dtype=torch.int32).t().contiguous()


class Engine:
    def __init__(self, state_dict, device, precision="bf16", chunk=None, frontend=None, mlp=None):
        self.lib = N.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise N.NativeError("the B200 engine needs a CUDA device; there is no CPU path")
        with torch.cuda.device(self.device):
            if not self.lib.acx_device_ok():
                raise N.NativeError(N.last_error())
        self.precision = precision
        self.w = PackedWeights(state_dict, self.device, precision)
        self.adt = N.ACX_BF16 if precision == "bf16" else N.ACX_F32
        self.esize = 2 if precision == "bf16" else 4
        self.chunk = int(chunk or os.environ.get("ACX_CHUNK", 64 if precision == "bf16" else 4))
        # which implementation of the two fusable pieces to run (both are libacx kernels)
        # front end: "fused" = the dense tensor-core kernel (default), "folded" = tensor-core kernel on folded frames (half the
        # DFT work, 0.355 vs 0.419 ms per 64 clips with its prep pass; needs the real-input symmetry of the loaded STFT rows.
        # Opt-in: on tonal / real audio the log-mel error against the reference grows from p99 9e-4 dB to 2.6e-3 dB -- past the
        # 1e-3 dB the parity tests assert; DESIGN.md k2), "simt" = fp32 CUDA cores
        self.frontend = frontend or os.environ.get("ACX_FRONTEND", "fused" if precision == "bf16" else "simt")
        if self.frontend == "folded" and getattr(self.w, "dftf", None) is None:
            self.frontend = "fused"
        self.mlp = mlp or os.environ.get("ACX_MLP", "fused")
        # depthwise 7x7: "tc" = banded-Toeplitz tcgen05 GEMMs (dwconv_tc.cu) + LayerNorm pass, "simt" = CUDA-core kernel
        # with the LayerNorm fused; ACX_DWCONV_TC_STAGES picks the stages that take the tensor-core route
        self.dwconv = os.environ.get("ACX_DWCONV", "tc" if precision == "bf16" else "simt")
        self.dwconv_tc_stages = tuple(int(c) for c in os.environ.get("ACX_DWCONV_TC_STAGES", "012"))
        # stages 0 / 1 with the fused MLP keep their activations GROUP-PLANAR ([C/8][M][8]) between the stage's entry
        # and its downsample layer: the tensor-core conv then moves whole cache lines (dwconv_tc.cu); ACX_GP=0 keeps NHWC
        self.gp = os.environ.get("ACX_GP", "1") == "1"
        # where the Block's LayerNorm runs behind the tensor-core conv: "fused" = on the operand tile inside the fused
        # MLP kernel (stages 0-1), "pass" = acx_layernorm_rows over HBM (always for stages whose MLP is two GEMMs)
        self.ln_mode = os.environ.get("ACX_LN", "fused")
        # downsample layers behind a planar stage: "1" = one implicit-GEMM kernel (ds_fused.cu), "0" = ln_patchify + GEMM
        # which input widths take it: at C = 384 (109 row tiles, N = 768 in two halves that both repeat the gather) the
        # two-kernel form measured faster (66 vs 74 us per 64 clips), so the default is the two large layers
        self.ds_fused = os.environ.get("ACX_DS_FUSED", "1") == "1"
        self.ds_fused_widths = tuple(int(c) for c in os.environ.get("ACX_DS_FUSED_C", "96,192").split(",") if c)
        if precision == "fp32":
            self.frontend, self.mlp, self.dwconv = "simt", "gemm", "simt"
        # LRU of workspaces keyed by (clips, samples); each owns the CUDA graphs captured over its buffers, so a
        # variable-length extraction or a ragged last batch neither re-allocates nor re-captures per call
        self._ws = collections.OrderedDict()
        self.max_workspaces = int(os.environ.get("ACX_WORKSPACES", 4))
        self.graph_after = int(os.environ.get("ACX_GRAPH_AFTER", 2))   # capture a shape on its 2nd use, not its 1st
        self.use_graph = os.environ.get("ACX_GRAPH", "1") == "1" and precision == "bf16"
        self._prof = None
        self._prof_only = None
        self.launches = 0

    # ---- workspace ------------------------------------------------------------------------------
    def _workspace(self, n, L):
        key = (n, L)
        ws = self._ws.get(key)
        if ws is not None:
            self._ws.move_to_end(key)
            return ws
        T, hs = out_time_dims(L)
        dev = self.device
        adt = self.w.act_dtype
        ld_pad = (max(L + N_FFT, HOP * (T + 3)) + 7) // 8 * 8     # fused front end reads whole hops
        ws = dict(T=T, hs=hs, ld_pad=ld_pad)
        if self.frontend == "folded":
            ws["f_hi"] = torch.empty(n, T, N_FFT, device=dev, dtype=torch.float16)      # folded frames [E | O], scaled fp16 pairs
            ws["f_lo"] = torch.empty(n, T, N_FFT, device=dev, dtype=torch.float16)
        elif self.frontend == "fused":
            ws["wav_hi"] = torch.empty(n, ld_pad, device=dev, dtype=torch.float16)
            ws["wav_lo"] = torch.empty(n, ld_pad, device=dev, dtype=torch.float16)
        else:
            ws["wav_pad"] = torch.empty(n, ld_pad, device=dev, dtype=torch.float32)
            ws["spec"] = torch.empty(n * T, 2 * N_BINS, device=dev, dtype=torch.float32)
        ws["logmel"] = torch.empty(n, T, N_MELS, device=dev, dtype=torch.float32)
        m0 = n * hs[0] * 56
        pad = 128 * DIMS[1]        # slack for the 128-row padded planes of the group-planar layout (stages 0 / 1)
        ws["x"] = torch.empty(m0 * DIMS[0] + pad, device=dev, dtype=adt)
        ws["y"] = torch.empty(m0 * DIMS[0] + pad, device=dev, dtype=adt)
        ws["hid"] = torch.empty(m0 * 4 * DIMS[0], device=dev, dtype=adt)
        if self.precision == "bf16":
            ws["xg"] = torch.empty(m0 * DIMS[0] + pad, device=dev, dtype=adt)      # group-planar residual stream (stages 0 - 2)
            ws["stats"] = torch.empty(n * hs[2] * 14 + 128, 2, device=dev, dtype=torch.float32)   # stage 2: per-row (rstd, -mean rstd)
        ws["pooled"] = torch.empty(n, DIMS[3], device=dev, dtype=torch.float32)
        # static outputs so that a captured CUDA graph can be replayed for any caller-owned output tensor
        ws["scene"] = torch.empty(n, DIMS[3], device=dev, dtype=torch.float32)
        ws["logits"] = torch.empty(n, N_CLASSES, device=dev, dtype=torch.float32)
        ws["probs"] = torch.empty(n, N_CLASSES, device=dev, dtype=torch.float32)
        ws["frame"] = torch.empty(n, DIMS[3], hs[3], 7, device=dev, dtype=torch.float32)
        ws["valid"] = torch.empty(6 * n, device=dev, dtype=torch.int32)     # ragged batches: ragged_table of the chunk
        ws["offsets"] = torch.empty(n, device=dev, dtype=torch.int64)       # windows: each row's first sample in the recording
        ws["graphs"] = {}         # (n, trunk, head, frame) -> (CUDAGraph, launches per replay); dies with the buffers
        ws["uses"] = {}
        while len(self._ws) >= max(1, self.max_workspaces):
            self._ws.popitem(last=False)          # least recently used shape (its graphs go with it)
        self._ws[key] = ws
        return ws

    # ---- per-kernel device timing (tools/time_stages.py, bench.py roofline leg) ------------------------
    def _call(self, tag, name, *args):
        self.launches += 1
        if self._prof is None or (self._prof_only is not None and not tag.startswith(self._prof_only)):
            N.call(name, *args)
            return
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        N.call(name, *args)
        e1.record()
        self._prof.append((tag, e0, e1))

    def _call_v(self, tag, name, valid, *args):
        """`name`, or with a per-clip bound (device pointer `valid`) its _ragged twin, which takes it before the stream."""
        if valid:
            self._call(tag, name + "_ragged", *args[:-1], valid, args[-1])
        else:
            self._call(tag, name, *args)

    def profile(self, wave, want=("logits",)):
        """Run once with a CUDA-event pair around every kernel launch (serialised on the current
        stream); returns [(tag, milliseconds)] in launch order."""
        self.start_timing(None)
        self.run(wave, want)
        return self.stop_timing()

    def start_timing(self, only=None):
        """Record a CUDA-event pair around every launch whose tag starts with `only` (all if None)."""
        self._prof, self._prof_only = [], only

    def stop_timing(self):
        torch.cuda.synchronize(self.device)
        res = [(tag, e0.elapsed_time(e1)) for tag, e0, e1 in self._prof]
        self._prof, self._prof_only = None, None
        return res

    def algorithmic_work(self, tag, n, L):
        """Roofline numerator of ONE launch of kernel `tag` on a chunk of n clips (SURVEY.md 8d):
        ("tensor", FLOPs) for the GEMM kernels, ("hbm", bytes) for the bandwidth kernels -- each activation
        tensor counted once per producing / consuming kernel, split-precision passes counted once."""
        T, hs = out_time_dims(L)
        es = self.esize
        if tag.startswith("ds_fused_c"):      # x read once, the stage's input written once; the patch matrix never exists
            C = int(tag[len("ds_fused_c"):])
            s = DIMS.index(C)
            return "hbm", 1.0 * n * es * (hs[s] * (56 >> s) * C + hs[s + 1] * (28 >> s) * 2 * C)
        if tag.startswith(("pw1_gelu", "pw2_resid", "ds_")):
            K, Nn = (int(t[1:]) for t in tag.split("_")[-2:])
            C = {"pw1_gelu": K, "pw2_resid": Nn, "ds": K // 4}[tag.rsplit("_", 2)[0]]
            s = DIMS.index(C)
            M = n * (hs[s + 1] * (28 >> s) if tag.startswith("ds_") else hs[s] * (56 >> s))
            return "tensor", 2.0 * M * Nn * K
        if tag.startswith("mlp_fused_c"):
            C = int(tag[len("mlp_fused_c"):])
            s = DIMS.index(C)
            return "tensor", 2.0 * (n * hs[s] * (56 >> s)) * C * 4 * C * 2
        if tag.startswith("row_stats_c"):
            C = int(tag.rsplit("_c", 1)[1])
            s = DIMS.index(C)
            return "hbm", 1.0 * n * hs[s] * (56 >> s) * C * es
        if tag.startswith(("dwconv_tc_c", "ln_rows_c", "to_gp_c")):
            C = int(tag.rsplit("_c", 1)[1])
            s = DIMS.index(C)
            return "hbm", 2.0 * n * hs[s] * (56 >> s) * C * es
        if tag.startswith("dwconv_ln_c"):
            C = int(tag[len("dwconv_ln_c"):])
            s = DIMS.index(C)
            return "hbm", 2.0 * n * hs[s] * (56 >> s) * C * es
        if tag.startswith("ln_patchify_c"):
            C = int(tag[len("ln_patchify_c"):])
            s = DIMS.index(C)
            return "hbm", 2.0 * n * hs[s] * (56 >> s) * C * es
        if tag in ("frontend_fused", "frontend_folded"):     # the REFERENCE's dense DFT + mel product, whatever the kernel does
            return "tensor", n * T * 2.0 * (N_FFT * 2 * N_BINS + N_BINS * N_MELS)
        if tag == "dft_simt":
            return "tensor", n * T * 2.0 * N_FFT * 2 * N_BINS
        if tag == "stem":
            return "hbm", n * (T * N_MELS * 4.0 + hs[0] * 56 * DIMS[0] * es)
        if tag == "frame_fold":
            return "hbm", n * L * 4.0 + n * T * N_FFT * 4.0
        if tag == "wave_prep":
            return "hbm", n * L * 4.0 + n * (L + N_FFT) * 4.0
        if tag == "head":
            return "hbm", n * hs[3] * 7 * DIMS[3] * es + N_CLASSES * DIMS[3] * 4.0
        return "hbm", 0.0

    # ---- stages (each is one libacx call) ----------------------------------------------------------
    def _wave_prep(self, wave, ws, n, L, st, rv=None, windows=False):
        """Reads the caller's tensor -> stays outside any captured graph.  rv: the ragged chunk's bound pointers or None.
        windows: `wave` is one 1-D recording and row b is its window at ws["offsets"][b] (the acx_*_windows forms)."""
        ld_pad = ws["ld_pad"]
        fn = "acx_wave_prep_pcm16" if wave.dtype == torch.int16 else "acx_wave_prep"
        if self.frontend == "folded":
            fn = "acx_frame_fold_pcm16" if wave.dtype == torch.int16 else "acx_frame_fold"
            args = (ws["f_hi"].data_ptr(), ws["f_lo"].data_ptr(), n, L, ws["T"], N_FFT, HOP)
            tag = "frame_fold"
        elif self.frontend == "fused":
            args = (ws["wav_hi"].data_ptr(), ws["wav_lo"].data_ptr(), n, L, N_FFT, ld_pad, N.ACX_BF16)
            tag = "wave_prep"
        else:
            args = (ws["wav_pad"].data_ptr(), 0, n, L, N_FFT, ld_pad, N.ACX_F32)
            tag = "wave_prep"
        if windows:
            self._call(tag, fn + "_windows", wave.data_ptr(), wave.numel(), ws["offsets"].data_ptr(), rv[0] if rv else 0,
                       *args, st)
        elif rv:
            self._call(tag, fn + "_ragged", wave.data_ptr(), *args, L, rv[0], st)   # rows of the (n, L) chunk are L samples apart
        else:
            self._call(tag, fn, wave.data_ptr(), *args, st)

    def _frontend(self, ws, n, L, st):
        w = self.w
        T, ld_pad = ws["T"], ws["ld_pad"]
        if self.frontend == "folded":
            self._call("frontend_folded", "acx_frontend_folded", ws["f_hi"].data_ptr(), ws["f_lo"].data_ptr(), w.dftf_hi.data_ptr(),
                       w.dftf_lo.data_ptr(), w.melc_hi.data_ptr(), w.melc_lo.data_ptr(), w.n_chunks, w.bn_scale.data_ptr(),
                       w.bn_shift.data_ptr(), ws["logmel"].data_ptr(), n, T, N_FFT, N_MELS, st)
        elif self.frontend == "fused":
            self._call("frontend_fused", "acx_frontend_fused", ws["wav_hi"].data_ptr(), ws["wav_lo"].data_ptr(), ld_pad,
                   w.dft_hi.data_ptr(), w.dft_lo.data_ptr(), w.melc_hi.data_ptr(), w.melc_lo.data_ptr(), w.n_chunks,
                   w.bn_scale.data_ptr(), w.bn_shift.data_ptr(), ws["logmel"].data_ptr(), n, T, N_FFT, HOP, N_MELS, st)
        else:
            self._call("dft_simt", "acx_gemm_f32", ws["wav_pad"].data_ptr(), ld_pad, T, HOP, w.dft_f32.data_ptr(),
                   ws["spec"].data_ptr(), 2 * N_BINS, n * T, 2 * N_BINS, N_FFT, N.EPI_BIAS, 0, 0, 0, st)
            self._call("power_mel_log", "acx_power_mel_log", ws["spec"].data_ptr(), 2 * N_BINS, N_BINS, w.melT.data_ptr(),
                   w.mel_lo.data_ptr(), w.mel_hi.data_ptr(), w.bn_scale.data_ptr(), w.bn_shift.data_ptr(),
                   ws["logmel"].data_ptr(), n * T, N_MELS, st)

    def _gemm(self, a, wt, out, M, Nn, K, epi, bias, gamma, resid, st):
        tag = f"{('ds', 'pw1_gelu', 'pw2_resid')[epi]}_k{K}_n{Nn}"
        if self.precision == "bf16":
            self._call(tag, "acx_gemm_bf16", a, wt, out, M, Nn, K, epi, bias, gamma, resid, st)
        else:
            self._call(tag, "acx_gemm_f32", a, M * K, M, K, wt, out, Nn, M, Nn, K, epi, bias, gamma, resid, st)

    def _trunk(self, ws, n, st, rv=None):
        w = self.w
        x, y, hid = ws["x"].data_ptr(), ws["y"].data_ptr(), ws["hid"].data_ptr()
        xgp = ws["xg"].data_ptr() if "xg" in ws else 0      # planar residual stream; trades places with y at a fused downsample
        # the stem writes stage 0's planar layout itself
        stem_gp = self.mlp == "fused" and self.dwconv == "tc" and 0 in self.dwconv_tc_stages and self.gp
        rT = rv[1] if rv else 0
        if stem_gp:
            self._call_v("stem", "acx_stem_gp", rT, ws["logmel"].data_ptr(), w.stem_w.data_ptr(), w.stem_b.data_ptr(),
                         w.stem_ln_w.data_ptr(), w.stem_ln_b.data_ptr(), xgp, n, ws["T"], N_MELS, st)
        else:
            self._call_v("stem", "acx_stem", rT, ws["logmel"].data_ptr(), w.stem_w.data_ptr(), w.stem_b.data_ptr(),
                         w.stem_ln_w.data_ptr(), w.stem_ln_b.data_ptr(), x, n, ws["T"], N_MELS, self.adt, st)
        Wd = 56
        entered_gp = False          # the previous downsample GEMM already wrote this stage's planar input
        for s in range(4):
            C, H = DIMS[s], ws["hs"][s]
            rh = rv[2 + s] if rv else 0         # ragged: each clip's own height at this stage
            M = n * H * Wd
            fused_mlp = self.mlp == "fused" and C in (96, 192)
            tc = self.dwconv == "tc" and s in self.dwconv_tc_stages
            gp = tc and fused_mlp and self.gp and Wd in (56, 28)
            gp2 = tc and not fused_mlp and self.gp and self.mlp == "fused" and Wd == 14 and C == 384   # planar, two-GEMM MLP
            if gp2:
                xg, vg = xgp, y
                if not entered_gp:
                    self._call(f"to_gp_c{C}", "acx_gp_transpose", x, xg, M, C, 1, st)
                stats = ws["stats"].data_ptr()
                for blk in w.blocks[s]:
                    self._call_v(f"dwconv_tc_c{C}", "acx_dwconv_tc_gp", rh, xg, blk["dw_w"].data_ptr(), blk["dw_b"].data_ptr(), vg, n, H, Wd, C, st)
                    self._call(f"row_stats_c{C}", "acx_gp_row_stats", vg, stats, M, C, st)
                    self._call(f"pw1_gelu_k{C}_n{4 * C}", "acx_gemm_bf16_pw1_gp", vg, blk["w1f"].data_ptr(), hid, M, 4 * C, C,
                               blk["b1f"].data_ptr(), stats, blk["s1"].data_ptr(), st)
                    self._call(f"pw2_resid_k{4 * C}_n{C}", "acx_gemm_bf16_pw2_gp", hid, blk["w2"].data_ptr(), xg, M, C, 4 * C,
                               blk["b2"].data_ptr(), blk["gamma"].data_ptr(), st)
            elif gp:
                # group-planar residual stream for this stage: xg <- x; the row-major x buffer becomes the conv output
                xg, vg = xgp, x
                if not (s == 0 and stem_gp) and not entered_gp:
                    self._call(f"to_gp_c{C}", "acx_gp_transpose", x, xg, M, C, 1, st)
            for blk in (() if gp2 else w.blocks[s]):
                if gp:
                    self._call_v(f"dwconv_tc_c{C}", "acx_dwconv_tc_gp", rh, xg, blk["dw_w"].data_ptr(), blk["dw_b"].data_ptr(), vg, n, H, Wd, C, st)
                    # the LayerNorm runs inside the MLP kernel: folded into pwconv1 as a rank-1 epilogue correction
                    # ("fused", default) or applied to the operand tile in shared memory (ACX_LN=smem)
                    if self.ln_mode == "smem":
                        self._call(f"mlp_fused_c{C}", "acx_mlp_fused_gp", vg, xg, blk["ln_w"].data_ptr(), blk["ln_b"].data_ptr(), 0,
                                   blk["w1"].data_ptr(), blk["b1"].data_ptr(), blk["w2"].data_ptr(), blk["b2"].data_ptr(),
                                   blk["gamma"].data_ptr(), M, C, st)
                    else:
                        self._call(f"mlp_fused_c{C}", "acx_mlp_fused_gp", vg, xg, 0, 0, blk["s1"].data_ptr(),
                                   blk["w1f"].data_ptr(), blk["b1f"].data_ptr(), blk["w2"].data_ptr(), blk["b2"].data_ptr(),
                                   blk["gamma"].data_ptr(), M, C, st)
                    continue
                ln_fused = False
                if tc:
                    self._call_v(f"dwconv_tc_c{C}", "acx_dwconv_tc", rh, x, blk["dw_w"].data_ptr(), blk["dw_b"].data_ptr(), y, n, H, Wd, C, st)
                    ln_fused = fused_mlp and self.ln_mode == "fused"
                    if not ln_fused:
                        self._call(f"ln_rows_c{C}", "acx_layernorm_rows", y, blk["ln_w"].data_ptr(), blk["ln_b"].data_ptr(), y, M, C, st)
                else:
                    self._call_v(f"dwconv_ln_c{C}", "acx_dwconv_ln", rh, x, blk["dw_w"].data_ptr(), blk["dw_b"].data_ptr(),
                                 blk["ln_w"].data_ptr(), blk["ln_b"].data_ptr(), y, n, H, Wd, C, self.adt, st)
                if ln_fused:
                    self._call(f"mlp_fused_c{C}", "acx_mlp_fused_ln", y, x, blk["ln_w"].data_ptr(), blk["ln_b"].data_ptr(),
                               blk["w1"].data_ptr(), blk["b1"].data_ptr(), blk["w2"].data_ptr(), blk["b2"].data_ptr(),
                               blk["gamma"].data_ptr(), M, C, st)
                elif fused_mlp:
                    self._call(f"mlp_fused_c{C}", "acx_mlp_fused", y, x, blk["w1"].data_ptr(), blk["b1"].data_ptr(), blk["w2"].data_ptr(),
                           blk["b2"].data_ptr(), blk["gamma"].data_ptr(), M, C, st)
                else:
                    self._gemm(y, blk["w1"].data_ptr(), hid, M, 4 * C, C, N.EPI_BIAS_GELU, blk["b1"].data_ptr(), 0, 0, st)
                    self._gemm(hid, blk["w2"].data_ptr(), x, M, C, 4 * C, N.EPI_BIAS_SCALE_RESID,
                               blk["b2"].data_ptr(), blk["gamma"].data_ptr(), x, st)
            if s < 3:
                d = w.ds[s]
                # the next stage takes its input group-planar: the downsample GEMM writes that layout itself
                entered_gp = (self.precision == "bf16" and self.mlp == "fused" and 2 * C in (96, 192, 384) and self.dwconv == "tc"
                              and (s + 1) in self.dwconv_tc_stages and self.gp and Wd // 2 in (56, 28, 14)
                              and os.environ.get("ACX_DS_GP", "1") == "1")
                if (gp or gp2) and self.ds_fused and C in self.ds_fused_widths:
                    # LayerNorm + 2x2 patch gather + GEMM in one kernel: the patch matrix never reaches HBM (ds_fused.cu)
                    self._call(f"ds_fused_c{C}", "acx_downsample_fused_gp", xg, d["ln_w"].data_ptr(), d["ln_b"].data_ptr(),
                               d["w_fused"].data_ptr(), d["b"].data_ptr(), y if entered_gp else x, n, H, Wd, C, 1 if entered_gp else 0, st)
                    if entered_gp:
                        xgp, y = y, xgp      # the kernel cannot write the planes it is still reading: the buffers trade places
                    Wd //= 2
                    continue
                if gp or gp2:
                    self._call(f"ln_patchify_c{C}", "acx_ln_patchify_gp", xg, d["ln_w"].data_ptr(), d["ln_b"].data_ptr(), y, n, H, Wd, C, st)
                else:
                    self._call(f"ln_patchify_c{C}", "acx_ln_patchify", x, d["ln_w"].data_ptr(), d["ln_b"].data_ptr(), y, n, H, Wd, C, self.adt, st)
                Wd //= 2
                Mo = n * ws["hs"][s + 1] * Wd
                if entered_gp:
                    self._call(f"ds_k{4 * C}_n{2 * C}", "acx_gemm_bf16_gp_out", y, d["w"].data_ptr(), xgp, Mo, 2 * C, 4 * C,
                               d["b"].data_ptr(), st)
                else:
                    self._gemm(y, d["w"].data_ptr(), x, Mo, 2 * C, 4 * C, N.EPI_BIAS, d["b"].data_ptr(), 0, 0, st)

    @staticmethod
    def _ragged_ptrs(ws, n, ragged):
        """Device pointers of the six rows of the chunk's (6, n) bound table in ws["valid"], or None."""
        if not ragged:
            return None
        base = ws["valid"].data_ptr()
        return [base + 4 * k * n for k in range(6)]

    def _body(self, ws, n, L, st, trunk, need_head, need_frame, ragged=False):
        """Everything after wave_prep for one chunk; writes only into the workspace (graph-capturable).  ragged: the
        kernels read each clip's bounds from ws["valid"] (data, so one graph serves every length mix)."""
        rv = self._ragged_ptrs(ws, n, ragged)
        self._frontend(ws, n, L, st)
        if not trunk:
            return
        self._trunk(ws, n, st, rv)
        x = ws["x"].data_ptr()
        h3 = ws["hs"][3]
        rh3 = rv[5] if rv else 0
        if need_head:
            w = self.w
            self._call_v("head", "acx_head", rh3, x, w.norm_w.data_ptr(), w.norm_b.data_ptr(), w.fc_w.data_ptr(),
                         w.fc_b.data_ptr(), ws["pooled"].data_ptr(), ws["scene"].data_ptr(), ws["logits"].data_ptr(),
                         ws["probs"].data_ptr(), n, h3, 7, DIMS[3], N_CLASSES, self.adt, st)
        if need_frame:
            self._call_v("frame_nchw", "acx_nhwc_to_nchw_f32", rh3, x, ws["frame"].data_ptr(), n, h3, 7, DIMS[3], self.adt, st)

    def _capture(self, ws, n, L, trunk, need_head, need_frame, ragged=False):
        """Capture the chunk's ~65 launches into one CUDA graph (fixed workspace pointers, tensor maps baked
        into the kernel parameters); one eager pass first so per-kernel attributes are already set."""
        st = torch.cuda.current_stream(self.device).cuda_stream
        before = self.launches
        self._body(ws, n, L, st, trunk, need_head, need_frame, ragged)
        per_replay = self.launches - before
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            cst = torch.cuda.current_stream(self.device).cuda_stream
            self._body(ws, n, L, cst, trunk, need_head, need_frame, ragged)
        self.launches = before                     # the eager pass is replaced by the first replay; capture launches nothing
        return g, per_replay

    # ---- public -----------------------------------------------------------------------------------
    def run(self, wave, want=("logits",), lengths=None):
        """wave: (B, L) float32 CUDA tensor (or int16 PCM, converted x / 32767. on the fly).  want: subset of {"logits", "scene", "frame", "logmel"}.
        Returns dict of fp32 tensors: probs/logits (B,527), scene (B,768), frame (B,768,T',7).

        lengths (B ints on the host, each in [MIN_RAGGED_LEN, L]): a ragged batch.  Clip b is wave[b, :lengths[b]] and its
        results equal a run of that clip alone; samples past it are never read, and frame rows past its own h3 are zero.
        Checked here, before any launch.  fp32 waveforms only; "logmel" is not available (its tail rows are not masked)."""
        assert wave.is_cuda and wave.dim() == 2 and wave.is_contiguous()
        assert wave.dtype in (torch.float32, torch.int16), "waveform must be float32 or int16 PCM"
        B, L = wave.shape
        T, hs = out_time_dims(L)
        if hs[3] < 1:
            raise ValueError(f"clip of {L} samples is too short for the 4-stage trunk")
        ragged = lengths is not None
        if ragged:
            lengths = check_lengths(lengths, B, L)
            if "logmel" in want:
                raise ValueError("a ragged batch has no log-mel output (its rows past each clip's end are not masked)")
            if wave.dtype != torch.float32:
                raise ValueError("a ragged batch takes a float32 waveform")
        dev = self.device
        out = {}
        need_head = "logits" in want or "scene" in want
        f32 = dict(device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            st = torch.cuda.current_stream(dev).cuda_stream
            if need_head:
                out["scene"] = torch.empty(B, DIMS[3], **f32)
                out["logits"] = torch.empty(B, N_CLASSES, **f32)
                out["probs"] = torch.empty(B, N_CLASSES, **f32)
            if "frame" in want:
                out["frame"] = torch.empty(B, DIMS[3], hs[3], 7, **f32)
            if "logmel" in want:
                out["logmel"] = torch.empty(B, T, N_MELS, **f32)
            for b0 in range(0, B, self.chunk):
                n = min(self.chunk, B - b0)
                ws = self._workspace(min(self.chunk, B), L)
                self._run_chunk(ws, n, L, st, want, lengths[b0:b0 + n] if ragged else None,
                                lambda rv: self._wave_prep(wave[b0:b0 + n], ws, n, L, st, rv))
                for name in ("logmel", "scene", "logits", "probs", "frame"):
                    if name in out:
                        out[name][b0:b0 + n].copy_(ws[name][:n])
        return out

    def _run_chunk(self, ws, n, L, st, want, lengths, prep):
        """One chunk of n clips on workspace ws (canvas L), the chunk loop body of run and run_windows: the ragged bound
        table when `lengths` (n ints) is given, then prep(rv) -- the prep launch, outside any graph because it reads the
        caller's buffer -- then everything after it, replayed from a CUDA graph or run eagerly.  Results stay in ws."""
        ragged = lengths is not None
        rv = None
        if ragged:
            # a fresh pinned host tensor per chunk: the caching host allocator keeps it until the copy has run
            tab = ragged_table(lengths).pin_memory()
            ws["valid"][:6 * n].view(6, n).copy_(tab, non_blocking=True)
            rv = self._ragged_ptrs(ws, n, True)
        prep(rv)
        need_head = "logits" in want or "scene" in want
        trunk = need_head or "frame" in want
        key = (n, L, trunk, need_head, "frame" in want, ragged)
        g = ws["graphs"].get(key) if (self.use_graph and self._prof is None) else None
        if g is None and self.use_graph and self._prof is None:
            ws["uses"][key] = ws["uses"].get(key, 0) + 1
            if ws["uses"][key] >= self.graph_after:      # a shape seen once (odd length, ragged tail) runs eagerly
                g = ws["graphs"][key] = self._capture(ws, n, L, *key[2:])
        if g is not None:
            g[0].replay()
            self.launches += g[1]
        else:
            self._body(ws, n, L, st, *key[2:])

    def run_windows(self, rec, plan, want=("logits",)):
        """Windows of one recording buffer, read in place.  rec: 1-D contiguous float32 or int16 PCM CUDA tensor (the
        recordings laid end to end); plan: windows.WindowPlan, whose `offset`s index rec.  Row i of every output equals a
        run of rec[offset_i : offset_i + length_i] alone.  Full-length windows run non-ragged on a canvas of plan.window,
        so they share run()'s workspace and CUDA graphs for that shape; own-length windows run ragged.  frame (N, 768,
        h3(plan.window), 7) has zeros past each window's own h3.  The plan is checked against rec before any launch."""
        from .windows import window_batches
        assert rec.is_cuda and rec.dim() == 1 and rec.is_contiguous()
        assert rec.dtype in (torch.float32, torch.int16), "recording must be float32 or int16 PCM"
        if "logmel" in want:
            raise ValueError("windows have no log-mel output")
        Nw, W = plan.length.numel(), int(plan.window)
        if Nw and not (int(plan.length.min()) >= MIN_RAGGED_LEN and int(plan.length.max()) <= W
                       and int(plan.offset.min()) >= 0 and int((plan.offset + plan.length).max()) <= rec.numel()):
            raise ValueError(f"window plan does not fit a recording buffer of {rec.numel()} samples "
                             f"(lengths must lie in [{MIN_RAGGED_LEN}, {W}] and every window inside the buffer)")
        batches = window_batches(plan, self.chunk)
        rows = {r: min(self.chunk, sum(len(idx) for _, ls, idx in batches if (ls is not None) == r)) for r in (False, True)}
        h3 = out_time_dims(W)[1][3]
        dev = self.device
        f32 = dict(device=dev, dtype=torch.float32)
        out = {}
        with torch.cuda.device(dev):
            st = torch.cuda.current_stream(dev).cuda_stream
            if "logits" in want or "scene" in want:
                out["scene"] = torch.empty(Nw, DIMS[3], **f32)
                out["logits"] = torch.empty(Nw, N_CLASSES, **f32)
                out["probs"] = torch.empty(Nw, N_CLASSES, **f32)
            if "frame" in want:
                out["frame"] = torch.empty(Nw, DIMS[3], h3, 7, **f32)
            for L, lengths, idx in batches:
                n = len(idx)
                ws = self._workspace(rows[lengths is not None], L)
                ws["offsets"][:n].copy_(plan.offset[idx].pin_memory(), non_blocking=True)
                self._run_chunk(ws, n, L, st, want, lengths, lambda rv: self._wave_prep(rec, ws, n, L, st, rv, windows=True))
                dst = torch.tensor(idx, dtype=torch.int64).to(dev, non_blocking=True)
                for name in ("scene", "logits", "probs"):
                    if name in out:
                        out[name].index_copy_(0, dst, ws[name][:n])
                if "frame" in out:
                    fr = ws["frame"][:n, :, :h3]               # a ragged canvas may have more rows than the window ...
                    if fr.shape[2] < h3:                       # ... or fewer: those are past every window's own h3
                        fr = torch.nn.functional.pad(fr, (0, 0, 0, h3 - fr.shape[2]))
                    out["frame"].index_copy_(0, dst, fr)
        return out
