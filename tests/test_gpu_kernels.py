"""GPU (B200): per-kernel parity of libacx (through the C ABI) against the CPU oracle."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from audioset_convnext_inf_b200 import _native as N          # noqa: E402
from oracle import convnext_oracle as O                       # noqa: E402
from oracle import weights                                    # noqa: E402

DEV = "cuda:0"


def _st():
    return torch.cuda.current_stream().cuda_stream


def _adt(dtype):
    return N.ACX_BF16 if dtype == torch.bfloat16 else N.ACX_F32


@pytest.fixture(scope="module")
def sd():
    return weights.make_state_dict("parity", 8)


def test_device_is_b200():
    assert N.load().acx_device_ok() == 1, N.last_error()


@pytest.mark.parametrize("pcm", [False, True])
@pytest.mark.parametrize("L", [320000, 1000, 40123])
def test_wave_prep_reflect_pad_and_split(L, pcm):
    """acx_wave_prep (fp32 input) and acx_wave_prep_pcm16 (int16 PCM, converted x / 32767 with one correct rounding):
    bit-exact reflect padding in fp32 mode, the scaled fp16 hi / lo split in bf16 mode."""
    w = weights.make_waveforms(2, n_samples=L, kind="tones", seed=2).to(DEV)
    entry = "acx_wave_prep"
    if pcm:
        wi = (w * 30000).round().clamp(-32768, 32767).to(torch.int16)
        wi[:, :3] = torch.tensor([-32768, 32767, 0], device=DEV, dtype=torch.int16)
        # utils/utilities.py:226 (true division), correctly rounded: IEEE fp32 division in numpy
        w = torch.from_numpy(wi.cpu().numpy().astype(np.float32) / np.float32(32767.0)).to(DEV)
        entry = "acx_wave_prep_pcm16"
    src = wi if pcm else w
    ld = (L + 1024 + 7) // 8 * 8
    ref = F.pad(w[:, None], (512, 512), mode="reflect")[:, 0]
    pad32 = torch.full((2, ld), 7.0, device=DEV)
    N.call(entry, src.data_ptr(), pad32.data_ptr(), 0, 2, L, 1024, ld, N.ACX_F32, _st())
    assert torch.equal(pad32[:, : L + 1024], ref)            # bit-exact copy
    assert (pad32[:, L + 1024:] == 0).all()
    hi = torch.empty(2, ld, device=DEV, dtype=torch.float16)       # fp16 pair of 2^8 * x (include/acx.h)
    lo = torch.empty_like(hi)
    N.call(entry, src.data_ptr(), hi.data_ptr(), lo.data_ptr(), 2, L, 1024, ld, N.ACX_BF16, _st())
    assert torch.equal(hi[:, : L + 1024], (ref * 256.0).to(torch.float16))
    rec = (hi.float() + lo.float()) / 256.0
    assert (rec[:, : L + 1024] - ref).abs().max() <= ref.abs().max() * 2.0 ** -21


@pytest.mark.parametrize("epi", [N.EPI_BIAS, N.EPI_BIAS_GELU, N.EPI_BIAS_SCALE_RESID])
@pytest.mark.parametrize("M,Nn,K", [(300, 192, 96), (1000, 1026, 1024), (130, 96, 384)])
def test_gemm_f32(M, Nn, K, epi):
    g = torch.Generator().manual_seed(M + Nn + K + epi)
    A = torch.randn(M, K, generator=g)
    W = torch.randn(Nn, K, generator=g) * 0.05
    bias, gamma, resid = torch.randn(Nn, generator=g), torch.rand(Nn, generator=g), torch.randn(M, Nn, generator=g)
    ref = A.double() @ W.double().t() + bias.double()
    if epi == N.EPI_BIAS_GELU:
        ref = F.gelu(ref)
    if epi == N.EPI_BIAS_SCALE_RESID:
        ref = resid.double() + gamma.double() * ref
    Ad, Wd, bd, gd, rd = (t.to(DEV) for t in (A, W, bias, gamma, resid))
    out = torch.empty(M, Nn, device=DEV)
    N.call("acx_gemm_f32", Ad.data_ptr(), 0, M, K, Wd.data_ptr(), out.data_ptr(), Nn, M, Nn, K, epi, bd.data_ptr(),
           gd.data_ptr(), rd.data_ptr(), _st())
    assert (out.cpu().double() - ref).abs().max() < 2e-4


def test_gemm_f32_overlapping_frames():
    """STFT framing: row t of clip b starts at b*ld + t*hop (torchlibrosa conv1d stride, CX:298)."""
    B, L, hop, K = 2, 6400, 320, 1024
    T = (L - K) // hop + 1
    wav = torch.randn(B, L)
    W = torch.randn(64, K) * 0.03
    frames = wav.unfold(1, K, hop)                            # (B, T, K)
    ref = frames.double() @ W.double().t()
    out = torch.empty(B * T, 64, device=DEV)
    wd, Wd = wav.to(DEV), W.to(DEV)
    N.call("acx_gemm_f32", wd.data_ptr(), L, T, hop, Wd.data_ptr(), out.data_ptr(), 64, B * T, 64, K, N.EPI_BIAS, 0, 0,
           0, _st())
    assert (out.cpu().double().view(B, T, 64) - ref).abs().max() < 1e-4


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_stem(sd, dtype):
    B, T = 2, 103
    lm = torch.randn(B, T, 224) * 2
    ref = O.stem(lm[:, None], sd, torch.float32).permute(0, 2, 3, 1)      # NHWC
    H0 = ref.shape[1]
    out = torch.empty(B, H0, 56, 96, device=DEV, dtype=dtype)
    w = sd["downsample_layers.0.0.weight"].reshape(96, 16).t().contiguous().to(DEV)
    args = [sd[k].to(DEV) for k in ("downsample_layers.0.0.bias", "downsample_layers.0.1.weight",
                                    "downsample_layers.0.1.bias")]
    lmd = lm.to(DEV)
    N.call("acx_stem", lmd.data_ptr(), w.data_ptr(), args[0].data_ptr(), args[1].data_ptr(), args[2].data_ptr(),
           out.data_ptr(), B, T, 224, _adt(dtype), _st())
    tol = 1e-4 if dtype == torch.float32 else 3e-2
    assert (out.float().cpu() - ref).abs().max() < tol


@pytest.mark.parametrize("B,T", [(1, 37), (8, 1001), (24, 1001)])
def test_stem_tensor_core_equals_cuda_core_up_to_one_bf16_ulp(sd, B, T):
    """bf16 mode runs the stem as a split-precision tcgen05 GEMM (stem_umma.cu), fp32 mode on the CUDA cores: the
    bf16 output must be the fp32 result rounded to bf16, give or take one ulp where the fp32 value sits on a rounding
    boundary.  (8 / 24 clips of 10 s = 882 / 2646 tiles: 2-6 tiles per persistent CTA, ragged last tile at T = 37.)"""
    g = torch.Generator().manual_seed(B * 1000 + T)
    lm = (torch.randn(B, T, 224, generator=g) * 2).to(DEV)
    H0 = (T + 4) // 4 + 1
    w = sd["downsample_layers.0.0.weight"].reshape(96, 16).t().contiguous().to(DEV)
    args = [sd[k].to(DEV) for k in ("downsample_layers.0.0.bias", "downsample_layers.0.1.weight",
                                    "downsample_layers.0.1.bias")]
    outs = {}
    for dtype in (torch.float32, torch.bfloat16):
        out = torch.empty(B, H0, 56, 96, device=DEV, dtype=dtype)
        N.call("acx_stem", lm.data_ptr(), w.data_ptr(), args[0].data_ptr(), args[1].data_ptr(), args[2].data_ptr(),
               out.data_ptr(), B, T, 224, _adt(dtype), _st())
        outs[dtype] = out
    torch.cuda.synchronize()
    ref = outs[torch.float32]
    got = outs[torch.bfloat16].float()
    ulp = torch.maximum(ref.abs(), torch.tensor(1e-30, device=DEV)).log2().floor().exp2() * 2.0 ** -7
    diff = (got - ref).abs()
    # the split-precision product carries ~16 operand bits, so ~1e-5 relative noise reaches the pre-rounding value and
    # about half a percent of the elements (those within that distance of a bf16 rounding boundary) round the other way
    assert (diff <= 0.5 * ulp * 1.02 + 2e-5).float().mean().item() > 0.99
    # never off by more than one ulp; next to zero (LayerNorm cancellation) the 16-bit operand split leaves an
    # ABSOLUTE noise of ~3e-5 (measured: 4 of 10.8 M elements between 2e-5 and 3e-5), far below bf16 resolution at |y| ~ 1
    assert (diff <= 1.01 * ulp + 1e-4).all()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("stage,H", [(0, 13), (1, 9), (2, 7), (3, 5), (3, 31)])
def test_dwconv_ln(sd, stage, H, dtype):
    C, Wd = O.DIMS[stage], 56 >> stage
    B = 2
    p = f"stages.{stage}.1."
    g = torch.Generator().manual_seed(stage * 100 + H)
    x = torch.randn(B, H, Wd, C, generator=g)
    xq = x.to(dtype)
    sdq = dict(sd)
    sdq[p + "dwconv.weight"] = sd[p + "dwconv.weight"].to(dtype).float()  # kernel holds taps in act dtype
    ref = O.block_dwconv_ln(xq.float().permute(0, 3, 1, 2), sdq, p, torch.float32)
    y = torch.empty(B, H, Wd, C, device=DEV, dtype=dtype)
    w = sd[p + "dwconv.weight"].reshape(C, 49).t().to(dtype).contiguous().to(DEV)
    b, lw, lb = (sd[p + k].to(DEV) for k in ("dwconv.bias", "norm.weight", "norm.bias"))
    xd = xq.to(DEV)
    N.call("acx_dwconv_ln", xd.data_ptr(), w.data_ptr(), b.data_ptr(), lw.data_ptr(), lb.data_ptr(), y.data_ptr(), B, H,
           Wd, C, _adt(dtype), _st())
    err = (y.float().cpu() - ref).abs().max().item()
    assert err < (2e-4 if dtype == torch.float32 else 4e-2), err


@pytest.mark.parametrize("stage,H,B", [(0, 13, 2), (0, 252, 3), (0, 130, 2), (1, 126, 2), (1, 9, 3), (2, 63, 3), (2, 64, 2),
                                       (3, 31, 2), (3, 5, 1)])
def test_dwconv_tc_then_layernorm_rows(sd, stage, H, B):
    """Tensor-core depthwise 7x7 (banded-Toeplitz tcgen05 GEMMs, acx_dwconv_tc) + acx_layernorm_rows against the
    oracle's F.conv2d / F.layer_norm (CX:76-78): full 10 s heights, heights that are not multiples of the 63-row tile,
    images shorter than the halo, every stage width.  The conv output is compared BEFORE the LayerNorm too: it is
    exact up to the bf16 rounding of the result (bf16 x bf16 products accumulate in fp32 in TMEM)."""
    C, Wd = O.DIMS[stage], 56 >> stage
    p = f"stages.{stage}.1."
    g = torch.Generator().manual_seed(stage * 1000 + H)
    xq = (torch.randn(B, H, Wd, C, generator=g) * 1.5).to(torch.bfloat16)
    wq = sd[p + "dwconv.weight"].to(torch.bfloat16)
    conv = F.conv2d(xq.float().permute(0, 3, 1, 2), wq.float(), sd[p + "dwconv.bias"], padding=3, groups=C)
    conv = conv.permute(0, 2, 3, 1).contiguous()
    ref = F.layer_norm(conv, (C,), sd[p + "norm.weight"], sd[p + "norm.bias"], 1e-6)
    w = wq.reshape(C, 49).t().contiguous().to(DEV)
    b, lw, lb = (sd[p + k].to(DEV) for k in ("dwconv.bias", "norm.weight", "norm.bias"))
    xd = xq.to(DEV)
    v = torch.full((B, H, Wd, C), float("nan"), device=DEV, dtype=torch.bfloat16)
    N.call("acx_dwconv_tc", xd.data_ptr(), w.data_ptr(), b.data_ptr(), v.data_ptr(), B, H, Wd, C, _st())
    torch.cuda.synchronize()
    vf = v.float().cpu()
    assert torch.isfinite(vf).all(), "unwritten outputs"
    spacing = 2.0 ** (torch.floor(torch.log2(conv.abs().clamp_min(2.0 ** -100))) - 7)     # bf16 spacing at |conv|
    assert ((vf - conv).abs() <= 0.51 * spacing + 1e-6).all(), ((vf - conv).abs() / spacing).max().item()
    y = torch.empty_like(v)
    N.call("acx_layernorm_rows", v.data_ptr(), lw.data_ptr(), lb.data_ptr(), y.data_ptr(), B * H * Wd, C, _st())
    err = (y.float().cpu() - ref).abs().max().item()
    assert err < 4e-2, err
    # in place
    N.call("acx_layernorm_rows", v.data_ptr(), lw.data_ptr(), lb.data_ptr(), v.data_ptr(), B * H * Wd, C, _st())
    assert torch.equal(v, y)


@pytest.mark.parametrize("stage,H,B", [(0, 13, 2), (0, 252, 3), (0, 130, 2), (1, 126, 2), (1, 9, 3), (1, 64, 1), (2, 63, 3),
                                       (2, 64, 2), (2, 6, 1)])
def test_dwconv_tc_group_planar(sd, stage, H, B):
    """acx_dwconv_tc_gp on the group-planar hand-off layout [C/8][B*H*W][8] (stages 0 / 1): bit-identical to the NHWC
    kernel (same MMAs, only the addressing differs), exact against F.conv2d up to the bf16 rounding of the result;
    acx_gp_transpose round-trips and equals the torch permutation; acx_ln_patchify_gp == acx_ln_patchify."""
    C, Wd = O.DIMS[stage], 56 >> stage
    p = f"stages.{stage}.2."
    g = torch.Generator().manual_seed(stage * 77 + H)
    xq = (torch.randn(B, H, Wd, C, generator=g) * 1.5).to(torch.bfloat16)
    wq = sd[p + "dwconv.weight"].to(torch.bfloat16)
    conv = F.conv2d(xq.float().permute(0, 3, 1, 2), wq.float(), sd[p + "dwconv.bias"], padding=3, groups=C)
    conv = conv.permute(0, 2, 3, 1).contiguous()
    w = wq.reshape(C, 49).t().contiguous().to(DEV)
    b = sd[p + "dwconv.bias"].to(DEV)
    xd = xq.to(DEV)
    M = B * H * Wd
    Mp = (M + 127) // 128 * 128                                   # plane stride: rows rounded up to 128
    xg = torch.zeros(C // 8, Mp, 8, device=DEV, dtype=torch.bfloat16)
    N.call("acx_gp_transpose", xd.data_ptr(), xg.data_ptr(), M, C, 1, _st())
    assert torch.equal(xg[:, :M], xd.view(M, C // 8, 8).permute(1, 0, 2)) and (xg[:, M:] == 0).all()
    vg = torch.full_like(xg, float("nan"))
    N.call("acx_dwconv_tc_gp", xg.data_ptr(), w.data_ptr(), b.data_ptr(), vg.data_ptr(), B, H, Wd, C, _st())
    v = torch.empty(B, H, Wd, C, device=DEV, dtype=torch.bfloat16)
    N.call("acx_gp_transpose", vg.data_ptr(), v.data_ptr(), M, C, 0, _st())
    v_nhwc = torch.empty_like(v)
    N.call("acx_dwconv_tc", xd.data_ptr(), w.data_ptr(), b.data_ptr(), v_nhwc.data_ptr(), B, H, Wd, C, _st())
    torch.cuda.synchronize()
    vf = v.float().cpu()
    assert torch.isfinite(vf).all(), "unwritten outputs"
    spacing = 2.0 ** (torch.floor(torch.log2(conv.abs().clamp_min(2.0 ** -100))) - 7)
    assert ((vf - conv).abs() <= 0.51 * spacing + 1e-6).all(), ((vf - conv).abs() / spacing).max().item()
    assert torch.equal(v, v_nhwc)
    if H % 2 == 0:
        lw, lb = sd[f"downsample_layers.{stage + 1}.0.weight"].to(DEV), sd[f"downsample_layers.{stage + 1}.0.bias"].to(DEV)
        a0 = torch.empty(M // 4, 4 * C, device=DEV, dtype=torch.bfloat16)
        a1 = torch.empty_like(a0)
        N.call("acx_ln_patchify", xd.data_ptr(), lw.data_ptr(), lb.data_ptr(), a0.data_ptr(), B, H, Wd, C, N.ACX_BF16, _st())
        N.call("acx_ln_patchify_gp", xg.data_ptr(), lw.data_ptr(), lb.data_ptr(), a1.data_ptr(), B, H, Wd, C, _st())
        assert torch.equal(a0, a1)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("stage,H", [(0, 10), (1, 7), (2, 63)])
def test_ln_patchify_then_gemm_is_downsample(sd, stage, H, dtype):
    C, Wd = O.DIMS[stage], 56 >> stage
    B = 2
    i = stage + 1
    x = torch.randn(B, H, Wd, C, generator=torch.Generator().manual_seed(i))
    xq = x.to(dtype)
    ref = O.downsample(xq.float().permute(0, 3, 1, 2), sd, i, torch.float32).permute(0, 2, 3, 1)   # (B,Ho,Wo,2C)
    Ho, Wo = H // 2, Wd // 2
    a = torch.empty(B * Ho * Wo, 4 * C, device=DEV, dtype=dtype)
    lw, lb = sd[f"downsample_layers.{i}.0.weight"].to(DEV), sd[f"downsample_layers.{i}.0.bias"].to(DEV)
    xd = xq.to(DEV)
    N.call("acx_ln_patchify", xd.data_ptr(), lw.data_ptr(), lb.data_ptr(), a.data_ptr(), B, H, Wd, C, _adt(dtype), _st())
    # patch matrix itself == LayerNorm'd pixels gathered (dy, dx, c)
    ln = O.layernorm_cf(xq.float().permute(0, 3, 1, 2), sd[f"downsample_layers.{i}.0.weight"],
                        sd[f"downsample_layers.{i}.0.bias"]).permute(0, 2, 3, 1)[:, : Ho * 2, : Wo * 2]
    pat = ln.reshape(B, Ho, 2, Wo, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(B * Ho * Wo, 4 * C)
    assert (a.float().cpu() - pat).abs().max() < (1e-4 if dtype == torch.float32 else 4e-2)
    w = sd[f"downsample_layers.{i}.1.weight"].permute(0, 2, 3, 1).reshape(2 * C, 4 * C).contiguous()
    out = (a.float().cpu() @ w.t() + sd[f"downsample_layers.{i}.1.bias"]).view(B, Ho, Wo, 2 * C)
    assert (out - ref).abs().max() < (1e-3 if dtype == torch.float32 else 6e-2)


@pytest.mark.parametrize("out_gp", [0, 1])
@pytest.mark.parametrize("stage,H,B", [(0, 10, 2), (0, 252, 3), (0, 7, 1), (1, 126, 2), (1, 9, 3), (2, 63, 3), (2, 6, 1), (2, 64, 5)])
def test_downsample_fused_implicit_gemm(sd, stage, H, B, out_gp):
    """acx_downsample_fused_gp (LayerNorm + 2x2/s2 patch gather + GEMM in one kernel, CX:230-235) against the oracle's
    downsample layer on the same bf16 input, and against the two-kernel form (acx_ln_patchify_gp + acx_gemm_bf16) it
    replaces; odd H (last row dropped), row counts that are not multiples of the 128-row tile, both output layouts."""
    from audioset_convnext_inf_b200.engine import pack_downsample_weight
    C, Wd = O.DIMS[stage], 56 >> stage
    i = stage + 1
    g = torch.Generator().manual_seed(100 * stage + H)
    xq = (torch.randn(B, H, Wd, C, generator=g) * 1.3 + 0.2).to(torch.bfloat16)
    ref = O.downsample(xq.float().permute(0, 3, 1, 2), sd, i, torch.float32).permute(0, 2, 3, 1)   # (B, Ho, Wo, 2C)
    Ho, Wo = H // 2, Wd // 2
    M, Mo = B * H * Wd, B * Ho * Wo
    Mp, Mop = (M + 127) // 128 * 128, (Mo + 127) // 128 * 128
    xg = torch.zeros(C // 8, Mp, 8, device=DEV, dtype=torch.bfloat16)
    xg[:, :M] = xq.to(DEV).view(M, C // 8, 8).permute(1, 0, 2)
    lw, lb = sd[f"downsample_layers.{i}.0.weight"].to(DEV), sd[f"downsample_layers.{i}.0.bias"].to(DEV)
    w4 = sd[f"downsample_layers.{i}.1.weight"]
    bias = sd[f"downsample_layers.{i}.1.bias"].to(DEV)
    wf = pack_downsample_weight(w4).to(torch.bfloat16).contiguous().to(DEV)
    if out_gp:
        outg = torch.full((2 * C // 8, Mop, 8), float("nan"), device=DEV, dtype=torch.bfloat16)
        N.call("acx_downsample_fused_gp", xg.data_ptr(), lw.data_ptr(), lb.data_ptr(), wf.data_ptr(), bias.data_ptr(),
               outg.data_ptr(), B, H, Wd, C, 1, _st())
        out = outg[:, :Mo].permute(1, 0, 2).reshape(Mo, 2 * C)
    else:
        out = torch.full((Mo + 3, 2 * C), float("nan"), device=DEV, dtype=torch.bfloat16)
        N.call("acx_downsample_fused_gp", xg.data_ptr(), lw.data_ptr(), lb.data_ptr(), wf.data_ptr(), bias.data_ptr(),
               out.data_ptr(), B, H, Wd, C, 0, _st())
        torch.cuda.synchronize()
        assert torch.isnan(out[Mo:].float()).all(), "wrote past the last output row"
        out = out[:Mo]
    # the two-kernel form on the same input
    a = torch.empty(Mo, 4 * C, device=DEV, dtype=torch.bfloat16)
    N.call("acx_ln_patchify_gp", xg.data_ptr(), lw.data_ptr(), lb.data_ptr(), a.data_ptr(), B, H, Wd, C, _st())
    wk = w4.permute(0, 2, 3, 1).reshape(2 * C, 4 * C).to(torch.bfloat16).contiguous().to(DEV)
    out2 = torch.empty(Mo, 2 * C, device=DEV, dtype=torch.bfloat16)
    N.call("acx_gemm_bf16", a.data_ptr(), wk.data_ptr(), out2.data_ptr(), Mo, 2 * C, 4 * C, N.EPI_BIAS, bias.data_ptr(), 0, 0, _st())
    torch.cuda.synchronize()
    of = out.float().cpu()
    assert torch.isfinite(of).all(), "unwritten outputs"
    err = (of - ref.reshape(Mo, 2 * C)).abs().max().item()
    assert err < 6e-2, err                                    # the bound test_ln_patchify_then_gemm_is_downsample uses (bf16)
    d2 = (of - out2.float().cpu()).abs()
    assert d2.max().item() < 3.2e-2 and d2.mean().item() < 1e-3, (d2.max().item(), d2.mean().item())


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("H", [31, 9, 1, 2, 3])
def test_head_and_frame_layout(sd, H, dtype):
    B = 3
    x = torch.randn(B, H, 7, 768, generator=torch.Generator().manual_seed(H))
    xq = x.to(dtype)
    scene_ref, logits_ref, probs_ref = O.pool_head(xq.float().permute(0, 3, 1, 2), sd, torch.float32)
    xd = xq.to(DEV)
    scene = torch.empty(B, 768, device=DEV)
    logits = torch.empty(B, 527, device=DEV)
    probs = torch.empty(B, 527, device=DEV)
    t = [sd[k].to(DEV) for k in ("norm.weight", "norm.bias", "head_audioset.weight", "head_audioset.bias")]
    pooled = torch.empty(B, 768, device=DEV)
    N.call("acx_head", xd.data_ptr(), t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(),
           pooled.data_ptr(), scene.data_ptr(), logits.data_ptr(), probs.data_ptr(), B, H, 7, 768, 527, _adt(dtype), _st())
    assert (scene.cpu() - scene_ref).abs().max() < 1e-4
    assert (logits.cpu() - logits_ref).abs().max() < 2e-4
    assert (probs.cpu() - probs_ref).abs().max() < 1e-4
    frame = torch.empty(B, 768, H, 7, device=DEV)
    N.call("acx_nhwc_to_nchw_f32", xd.data_ptr(), frame.data_ptr(), B, H, 7, 768, _adt(dtype), _st())
    assert torch.equal(frame.cpu(), xq.float().permute(0, 3, 1, 2))


def test_frontend_fp32_path_logmel(sd):
    """SIMT front end (fp32-accurate mode) vs the oracle's torchlibrosa restatement (CX:298-306)."""
    import audioset_convnext_inf_b200 as acx
    m = acx.convnext_tiny(drop_path_rate=0.0, after_stem_dim=[252, 56])
    m.load_state_dict(sd)
    m = m.to(DEV).eval().set_precision("fp32")
    for kind in ("noise", "tones"):
        w = weights.make_waveforms(2, n_samples=64000, kind=kind, seed=4)
        ref = O.frontend(w, sd, torch.float32)
        ref64 = O.frontend(w, sd, torch.float64)
        got = m.forward_logmel(w.to(DEV)).cpu()
        err = (got - ref).abs()
        err64 = (got.double() - ref64).abs().max().item()
        ref_err64 = (ref.double() - ref64).abs().max().item()
        print(f"[{kind}] logmel_bn |ours-ref| max {err.max():.3e} mean {err.mean():.3e}; vs fp64: ours {err64:.3e} ref {ref_err64:.3e}")
        # bn0 scales dB by ~1/20: 1e-3 dB abs -> 5e-5 normalised; allow the reference's own fp32 noise
        assert err64 < max(3 * ref_err64, 1e-4)


@pytest.mark.parametrize("L", [64000, 40123, 700])
@pytest.mark.parametrize("pcm", [False, True])
def test_frame_fold_matches_reflect_padded_frames(L, pcm):
    """acx_frame_fold: F[b, t, :512] = E, F[b, t, 512:] = O of the reflect-padded frame t (center=True, hop 320), folded in
    fp32 and carried as a 2^8-scaled fp16 pair: hi + lo reproduces the fp32 fold to the pair's 22 bits."""
    B, T = 2, L // 320 + 1
    w = weights.make_waveforms(B, n_samples=L, kind="tones", seed=9)
    if pcm:
        wi = (w * 20000).round().clamp(-32768, 32767).to(torch.int16)
        w = wi.float() / 32767.0                                              # utils/utilities.py:226 (true division)
    xp = F.pad(w[:, None], (512, 512), mode="reflect")[:, 0]
    fr = xp.unfold(1, 1024, 320)[:, :T]                                        # (B, T, 1024)
    mir = torch.arange(1023, 512, -1)
    E = torch.cat([fr[..., 512:513], fr[..., 1:512] + fr[..., mir]], -1)
    Od = torch.cat([torch.zeros_like(fr[..., :1]), fr[..., 1:512] - fr[..., mir]], -1)
    ref = torch.cat([E, Od], -1)
    hi = torch.full((B, T, 1024), float("nan"), device=DEV, dtype=torch.float16)
    lo = torch.full_like(hi, float("nan"))
    src = (wi if pcm else w).to(DEV)
    N.call("acx_frame_fold_pcm16" if pcm else "acx_frame_fold", src.data_ptr(), hi.data_ptr(), lo.data_ptr(), B, L, T, 1024, 320, _st())
    got = ((hi.float() + lo.float()) / 256.0).cpu()
    assert torch.isfinite(got).all()
    assert (got - ref).abs().max().item() < 2.0 ** -20 * max(1.0, ref.abs().max().item())


def test_dft_fold_needs_symmetric_rows(sd):
    """engine.fold_dft_weights: the periodic-Hann STFT rows of the checkpoint fold (and reproduce the dense product); rows
    without the real-input symmetry are refused, and the engine then keeps the dense kernel."""
    import audioset_convnext_inf_b200 as acx
    from audioset_convnext_inf_b200.engine import fold_dft_weights
    cr = sd["spectrogram_extractor.stft.conv_real.weight"][:, 0, :].float()
    ci = sd["spectrogram_extractor.stft.conv_imag.weight"][:, 0, :].float()
    f = fold_dft_weights(cr, ci, 7)
    assert f is not None and f.shape == (4 * 256, 512)
    x = torch.randn(3, 1024, dtype=torch.float64)
    mir = torch.arange(1023, 512, -1)
    E = torch.cat([x[:, 512:513], x[:, 1:512] + x[:, mir]], 1)
    Od = torch.cat([torch.zeros(3, 1, dtype=torch.float64), x[:, 1:512] - x[:, mir]], 1)
    fr = f.double().view(4, 4, 64, 512)
    for c in range(7):
        assert (E @ fr[c // 2, c % 2].t() - x @ cr.double()[64 * c:64 * c + 64].t()).abs().max() < 1e-4
        assert (Od @ fr[c // 2, 2 + c % 2].t() - x @ ci.double()[64 * c:64 * c + 64].t()).abs().max() < 1e-4
    bad = cr.clone()
    bad[5, 100] += 1e-3
    assert fold_dft_weights(bad, ci, 7) is None
    sd2 = dict(sd)
    sd2["spectrogram_extractor.stft.conv_real.weight"] = bad[:, None, :].clone()
    m = acx.convnext_tiny(drop_path_rate=0.0, after_stem_dim=[252, 56])
    m.load_state_dict(sd2)
    m = m.to(DEV).eval().set_precision("bf16")
    assert m._get_engine().frontend == "fused"
    w = weights.make_waveforms(1, n_samples=32000, kind="noise", seed=1)
    assert (m.forward_logmel(w.to(DEV)).cpu() - O.frontend(w, sd2, torch.float32)).abs().max() < 1e-3


@pytest.mark.parametrize("frontend", ["folded", "fused"])
@pytest.mark.parametrize("kind,L", [("noise", 64000), ("tones", 64000), ("tones", 320000), ("tones", 40123)])
def test_frontend_fused_logmel(sd, kind, L, frontend, monkeypatch):
    """tcgen05 front end (split-fp16 x3 DFT -- on folded frames by default, dense with ACX_FRONTEND=fused -- and split-bf16
    x3 mel GEMM) vs the oracle's torchlibrosa restatement.
    Metrics per SURVEY.md Appendix C; values are in bn0-normalised units (1 unit ~ 20 dB here)."""
    import audioset_convnext_inf_b200 as acx
    monkeypatch.setenv("ACX_FRONTEND", frontend)
    m = acx.convnext_tiny(drop_path_rate=0.0, after_stem_dim=[252, 56])
    m.load_state_dict(sd)
    m = m.to(DEV).eval().set_precision("bf16")
    assert m._get_engine().frontend == frontend
    w = weights.make_waveforms(2, n_samples=L, kind=kind, seed=4)
    ref = O.frontend(w, sd, torch.float32)
    ref64 = O.frontend(w, sd, torch.float64)
    got = m.forward_logmel(w.to(DEV)).cpu()
    assert got.shape == ref.shape
    err = (got.double() - ref64).abs()
    ref_err = (ref.double() - ref64).abs()
    # bins within 80 dB of the clip maximum (un-normalised dB = before bn0)
    raw = O.logmel(O.spectrogram(w, sd, torch.float64), sd, torch.float64)
    mask = raw > raw.amax(dim=(1, 2), keepdim=True) - 80.0
    print(f"[{frontend} {kind} L={L}] vs fp64: max {err.max():.3e} mean {err.mean():.3e} p99 {err.flatten().quantile(0.99):.3e} "
          f"masked-max {err[mask].max():.3e} | reference fp32 vs fp64: max {ref_err.max():.3e} mean {ref_err.mean():.3e}")
    assert torch.isfinite(got).all()
    # scaled fp16 pairs keep 22 operand bits: the front end sits within ~2x of the reference's OWN fp32 rounding noise
    # (measured: noise mean 1.4e-6 / max 5e-5; adversarial tones over a -80 dB floor mean 2.2e-5 / in-band max 4e-4,
    # reference fp32 vs fp64 mean 1.6e-5 / max 5.5e-3).  The first, bf16-pair version was 40x worse on the tones.
    lim = dict(noise=(1e-5, 3e-4, 3e-5), tones=(1e-4, 2e-3, 1e-3))[kind]
    assert err.max() < 4 * ref_err.max() + 1e-3
    assert err.mean() < lim[0] and err[mask].max() < lim[1] and err.flatten().quantile(0.99) < lim[2]


def test_c_abi_rejects_bad_arguments_with_messages():
    """Error convention of the boundary: non-zero code + thread-local message, nothing launched, no exception in C."""
    lib = N.load()
    t = torch.zeros(64, device=DEV)
    p = t.data_ptr()
    assert lib.acx_dwconv_ln(p, p, p, p, p, p, 1, 8, 10, 96, N.ACX_BF16, 0) != 0 and "multiple of 7" in N.last_error()
    assert lib.acx_dwconv_ln(p, p, p, p, p, p, 1, 8, 14, 100, N.ACX_BF16, 0) != 0 and "unsupported channel" in N.last_error()
    assert lib.acx_dwconv_ln(0, p, p, p, p, p, 1, 8, 14, 96, N.ACX_BF16, 0) != 0 and "null" in N.last_error()
    assert lib.acx_ln_patchify(p, p, p, p, 1, 8, 14, 100, N.ACX_BF16, 0) != 0 and "unsupported shape" in N.last_error()
    assert lib.acx_wave_prep(p, p, p, 1, 100, 1024, 2048, N.ACX_BF16, 0) != 0 and "reflect" in N.last_error()
    assert lib.acx_wave_prep(p, p, p, 1, 2000, 1024, 2000, N.ACX_BF16, 0) != 0 and "ld_pad" in N.last_error()
    assert lib.acx_frontend_fused(p, p, 4096, p, p, p, p, 7, p, p, p, 1, 1001, 512, 320, 224, 0) != 0
    assert "n_fft=1024" in N.last_error()
    assert lib.acx_frontend_folded(p, p, p, p, p, p, 7, p, p, p, 1, 1001, 512, 224, 0) != 0 and "n_fft=1024" in N.last_error()
    assert lib.acx_frame_fold(p, p, p, 1, 400, 2, 1024, 320, 0) != 0 and "reflect" in N.last_error()
    assert lib.acx_head(p, p, p, p, p, p, p, p, p, 1, 31, 7, 770, 527, N.ACX_BF16, 0) != 0 and "unsupported" in N.last_error()
    assert lib.acx_mlp_fused(p, p, p, p, p, p, p, 0, 96, 0) != 0 and "positive" in N.last_error()
    torch.cuda.synchronize()          # nothing above may have poisoned the context
