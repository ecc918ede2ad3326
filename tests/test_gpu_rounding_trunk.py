"""GPU (B200): rounding-level tests of the CUDA-core depthwise conv + LayerNorm (acx_dwconv_ln, acx_dwconv_ln_ragged) and of
the downsample layers (acx_ln_patchify, acx_ln_patchify_gp, acx_downsample_fused_gp).

Every bound is a formula of the kernel's documented arithmetic, against an fp64 reference computed on the device:
half an output ulp (bf16 outputs) + an fp32 term K u (magnitudes) whose K follows from the reduction depth, and on random
operands an aggregate limit on the fraction of outputs that differ from the round-to-nearest of the fp64 emulation.

* A  dwconv_ln LayerNorm readout: center tap 1, other taps 0, bias = a common fp32 offset mu, so every conv output is
     exactly v = fp32(x + mu) and the output is the kernel's LayerNorm of known values -- mu / sigma from 0 to 1000 (a
     single-pass variance cancels there), u^2 near eps, every strip configuration and both row-group paths of C = 768.
* B  dwconv_ln on random operands (heights below the halo, not multiples of the 4-row group, partial last block), and the
     ragged form against the clip run alone, bit for bit, with NaN past each clip's rows.
* C  ln_patchify (bf16, fp32) and ln_patchify_gp: every entry of the patch matrix against the fp64 LayerNorm.
* D  ds_fused: the bf16 A operand read out through selector conv weights (1 at one K entry per output column), at shapes
     where every persistent CTA runs three or more tiles (the next tile's statistics ride along the current tile's K
     blocks), and on random operands against an fp64 emulation of the operand rounding and the fp32 accumulation.
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from audioset_convnext_inf_b200 import _native as N          # noqa: E402

DEV = "cuda:0"
F64 = torch.float64
BF16 = torch.bfloat16
U24 = 2.0 ** -24                       # fp32 unit roundoff
NAN = float("nan")


def _st():
    return torch.cuda.current_stream().cuda_stream


def _adt(dtype):
    return N.ACX_BF16 if dtype == BF16 else N.ACX_F32


# ---- fp64 models of the roundings (as in test_gpu_rounding.py) ---------------------------------------------------------
def _ulp(v):
    """bf16 spacing at |v| (normal range)."""
    return torch.exp2(torch.floor(torch.log2(v.abs().clamp_min(2.0 ** -126))) - 7)


def _rn(v):
    """fp64 -> nearest bf16 value (ties to even), without a detour through fp32."""
    q = _ulp(v)
    return torch.round(v / q) * q


def _to_gp_nan(t):
    """(M, C) -> group-planar [C/8][Mp][8], Mp = M rounded up to 128, the padding rows M..Mp NaN."""
    M, C = t.shape
    Mp = (M + 127) // 128 * 128
    out = torch.full((C // 8, Mp, 8), NAN, device=t.device, dtype=t.dtype)
    out[:, :M] = t.view(M, C // 8, 8).permute(1, 0, 2)
    return out


def _ln64(v):
    """fp64 LayerNorm statistics over the last dim (eps 1e-6): mean, d = v - mean, rstd."""
    mean = v.mean(-1, keepdim=True)
    d = v - mean
    rstd = 1.0 / torch.sqrt((d * d).mean(-1, keepdim=True) + 1e-6)
    return mean, d, rstd


# ---- LayerNorm input rows --------------------------------------------------------------------------------------------
# (mean, u): +-u alternating by channel, every value bf16-exact (statistics exact in fp32); u^2 comparable to eps = 1e-6
CLOSED_ROWS = [(0.0, 2.0 ** -10), (0.0, 2.0 ** -11), (0.0, 2.0 ** -9), (0.0, 0.5), (64.0, 0.5), (-96.0, 0.5),
               (8.0, 2.0 ** -4), (1.0, 2.0 ** -7)]
# (mean, sigma): mean + sigma N(0, 1) rounded to the input type, mean / sigma from 64 to 400: the sums of these rows round,
# and an unshifted single-pass variance loses 1e-3 .. 1e-2 of rstd to cancellation
OFFSET_ROWS = [(16.0, 0.25), (64.0, 0.5), (128.0, 1.0), (100.0, 0.25), (-48.0, 0.125), (3.0, 0.0234375)]
# sigma N(0, 1) with sigma^2 near eps
EPS_ROWS = [(0.0, 1e-3), (0.0, 7e-4), (0.0, 2e-3)]


def _ln_rows(P, C, dtype, seed, far_first=False):
    """(P, C) input rows in `dtype`, the families above cycling by row.  far_first: one more offset family whose first
    channel sits 8 sigma from the row's mean (the kernels that shift by the first channel lose the most there; the error
    stays bounded because (x0 - mean)^2 <= C var)."""
    g = torch.Generator().manual_seed(seed)
    fams = [("c", r) for r in CLOSED_ROWS] + [("o", r) for r in OFFSET_ROWS] + [("o", r) for r in EPS_ROWS]
    if far_first:
        fams += [("f", r) for r in OFFSET_ROWS[:4]]
    rows = torch.empty(P, C, dtype=F64)
    sign = 1.0 - 2.0 * (torch.arange(C) % 2).to(F64)
    z = torch.randn(P, C, generator=g, dtype=F64)
    for i, (kind, (mu, s)) in enumerate(fams):
        sel = torch.arange(i, P, len(fams))
        if kind == "c":
            rows[sel] = mu + s * sign
        else:
            rows[sel] = mu + s * z[sel]
            if kind == "f":
                rows[sel, 0] = mu + 8.0 * s
    return rows.to(dtype).to(DEV)


def _affine(C, seed):
    g = torch.Generator().manual_seed(seed)
    lw = (torch.rand(C, generator=g) * 1.2 + 0.3) * torch.where(torch.rand(C, generator=g) < 0.1, -1.0, 1.0)
    lb = torch.randn(C, generator=g) * 0.2
    return lw.to(DEV), lb.to(DEV)


def _check(tag, got, ref, bound, bf16, frac_limit=None):
    """|got - ref| <= bound (+ half a bf16 ulp of got); optionally the fraction of outputs != RN(ref) below frac_limit."""
    assert torch.isfinite(got).all(), f"{tag}: unwritten or non-finite outputs"
    if bf16:
        bound = bound + 0.5 * _ulp(got)
    err = (got - ref).abs()
    ratio = (err / bound).max().item()
    frac = (got != _rn(ref)).double().mean().item() if bf16 else 0.0
    print(f"  {tag}: max |err| / bound {ratio:.3f}" + (f"; outputs != RN(ref) {100 * frac:.3f} %" if bf16 else ""))
    assert (err <= bound).all(), (tag, ratio)
    if frac_limit is not None:
        assert frac < frac_limit, (tag, frac)
    return frac


# ======================================================================================================================
# A / B.  dwconv_ln
# ======================================================================================================================
def _dw_K(C):
    """fp32 error of the kernel's LayerNorm, in units of u (|v| + mean|v|) rstd |ln_w|: each sum is a pair add, a 16-lane
    tree (4 levels) and C/32 - 1 group adds in a fixed order (depth C/32 + 4); + the 1/C scalings, the deviation, rsqrtf
    (2 ulp) and the affine step."""
    return C // 32 + 16


def _dw_shift_term(v, d, rstd, C):
    """The bf16 instantiation's single pass sums d = v - v0 and d^2 (v0 the pixel's first channel): with sums of depth
    C/32 + 4, the shifted mean errs by (C/32 + 6) u mean|v - v0| and the variance E[d^2] - E[d]^2 by (C/32 + 6) u E[d^2]
    relative to var + eps.  (Without the shift E[d^2] / var would be 1 + mean^2 / var.)  Returned in units of rstd |ln_w|."""
    D = C // 32 + 6
    sh = v - v[..., :1]
    E2 = (sh * sh).mean(-1, keepdim=True)
    return D * U24 * (0.5 * d.abs() * E2 * rstd ** 2 + sh.abs().mean(-1, keepdim=True))


def _dwconv(x, w49, bias, lw, lb, valid=None):
    """acx_dwconv_ln (valid None) or acx_dwconv_ln_ragged on x (B, H, W, C); the output starts as NaN."""
    B, H, W, C = x.shape
    y = torch.full_like(x, NAN)
    p = (x.data_ptr(), w49.data_ptr(), bias.data_ptr(), lw.data_ptr(), lb.data_ptr(), y.data_ptr(), B, H, W, C, _adt(x.dtype))
    if valid is None:
        N.call("acx_dwconv_ln", *p, _st())
    else:
        N.call("acx_dwconv_ln_ragged", *p, valid.data_ptr(), _st())
    return y


def _dw_bound(v, rstd, lw, lb, C, dv=None, shifted=False):
    """fp32 slack of dwconv_ln around the fp64 LayerNorm of v: K u (|v| + mean|v|) rstd |ln_w| + 2 u |ln_b| (+ the shifted
    single pass's term); with dv (a bound on |kernel conv - v| per element) the first-order propagation of dv through the
    LayerNorm: |d LN_i| <= rstd (dv_i + mean dv + |n_i| rms dv) |ln_w|."""
    aw = lw.double().abs()
    b = _dw_K(C) * U24 * (v.abs() + v.abs().mean(-1, keepdim=True)) * rstd * aw + 2 * U24 * lb.double().abs()
    if shifted:
        b = b + _dw_shift_term(v, v - v.mean(-1, keepdim=True), rstd, C) * rstd * aw
    if dv is not None:
        n = (v - v.mean(-1, keepdim=True)) * rstd
        b = b + 1.01 * rstd * aw * (dv + dv.mean(-1, keepdim=True) + n.abs() * dv.pow(2).mean(-1, keepdim=True).sqrt())
    return b


READOUT_MU = 77.3                            # common fp32 bias of the offset launch
READOUT_K = (8.0, 30.0, 100.0, 300.0, 1000.0)   # mu / sigma of its pixels


def _readout_input(B, H, W, C, dtype, mu, seed):
    """Pixels cycle through sigma families: for mu = 0 unit, 1e-3 and 2e-3 spreads and +-2^-10 / +-2^-9 rows (u^2 near eps);
    otherwise sigma = mu / k for k in READOUT_K.  x is bf16-valued (full mantissa) in either dtype."""
    g = torch.Generator().manual_seed(seed)
    P = B * H * W
    z = torch.randn(P, C, generator=g, dtype=F64)
    sign = 1.0 - 2.0 * (torch.arange(C) % 2).to(F64)
    if mu == 0.0:
        fams = [("n", 1.0), ("n", 1e-3), ("n", 2e-3), ("a", 2.0 ** -10), ("a", 2.0 ** -9)]
    else:
        fams = [("n", mu / k) for k in READOUT_K]
    x = torch.empty(P, C, dtype=F64)
    fam = torch.arange(P) % len(fams)
    for i, (kind, s) in enumerate(fams):
        sel = fam == i
        x[sel] = s * (z[sel] if kind == "n" else sign.expand(int(sel.sum()), C))
    return x.to(BF16).to(dtype).view(B, H, W, C).to(DEV), fam.view(B, H, W).to(DEV), fams


# (C, W, H, B): C = 96 with 4 and 2 strips per block, C = 192 with 2 and 1, C = 384, C = 768 with 4 row groups per block
# (H >= 13; H = 17 leaves the second block one group) and with one (H < 13)
DW_READOUT_SHAPES = [(96, 56, 5, 2), (96, 14, 9, 2), (192, 28, 6, 2), (192, 21, 7, 1), (384, 14, 5, 2), (768, 7, 13, 2),
                     (768, 7, 17, 1), (768, 7, 9, 2)]


@pytest.mark.parametrize("dtype", [BF16, torch.float32])
@pytest.mark.parametrize("C,W,H,B", DW_READOUT_SHAPES)
def test_dwconv_ln_layernorm_readout(C, W, H, B, dtype):
    """acx_dwconv_ln with the center tap 1 and every other tap 0: the conv output is exactly v = fp32(x + mu) (mu the
    common bias), so the output must be the fp64 LayerNorm of v within half an output ulp (bf16) plus
    K u (|v| + mean|v|) rstd |ln_w| + 2 u |ln_b| (+ the error of the bf16 form's statistics shifted by the first channel),
    for mu / sigma up to 1000 and for u^2 near eps.  An unshifted single pass fails from mu / sigma = 30 on."""
    w49 = torch.zeros(49, C, device=DEV)
    w49[24] = 1.0
    w49 = w49.to(dtype)
    lw, lb = _affine(C, seed=C + H)
    for mu in (0.0, READOUT_MU):
        x, fam, fams = _readout_input(B, H, W, C, dtype, mu, seed=C * 31 + H + int(mu))
        bias = torch.full((C,), mu, device=DEV, dtype=torch.float32)
        y = _dwconv(x, w49, bias, lw, lb).double()
        v = (x.float() + bias).double()                                 # the conv output, exact
        _, d, rstd = _ln64(v)
        ref = d * rstd * lw.double() + lb.double()
        bound = _dw_bound(v, rstd, lw, lb, C, shifted=dtype == BF16)
        err = (y - ref).abs() / (bound + (0.5 * _ulp(y) if dtype == BF16 else 0.0))
        per = [f"{k}{s:.3g}: {err[fam == i].max().item():.2f}" for i, (k, s) in enumerate(fams)]
        _check(f"dwconv_ln readout {dtype} C={C} W={W} H={H} mu={mu} [{', '.join(per)}]", y, ref, bound, dtype == BF16)


# Fraction of bf16 outputs that differ from the round-to-nearest of the fp64 emulation on random operands.  Measured on one
# NVIDIA B200 (1000 W power limit): at most 0.010 % without a bias offset and 0.064-0.163 % with it, every C and H.
FRAC_DW_LIMIT = 0.005


def _dw_random(B, H, W, C, dtype, offset, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, H, W, C, generator=g).to(BF16).to(dtype)
    w49 = (torch.randn(49, C, generator=g) * 0.12).to(BF16).to(dtype)
    bias = torch.randn(C, generator=g) * 0.02 + offset
    lw, lb = _affine(C, seed)
    return [t.to(DEV) for t in (x, w49, bias)] + [lw, lb]


def _conv64(x, w49, bias):
    """exact depthwise 7x7 (zero padding 3) in fp64 -> (B, H, W, C); with bias None the conv alone."""
    B, H, W, C = x.shape
    wk = w49.double().t().reshape(C, 1, 7, 7)
    out = F.conv2d(x.double().permute(0, 3, 1, 2), wk, None, padding=3, groups=C).permute(0, 2, 3, 1)
    return out if bias is None else out + bias.double()


@pytest.mark.parametrize("dtype", [BF16, torch.float32])
@pytest.mark.parametrize("C,W", [(96, 56), (192, 28), (384, 14), (768, 7)])
def test_dwconv_ln_emulated_rounding(C, W, dtype):
    """acx_dwconv_ln on random bf16-valued operands against the fp64 conv + LayerNorm: the conv accumulates 49 fp32 FMAs
    from the bias (|conv - exact| <= 50 u (|b| + sum |x w|)), which the LayerNorm propagates to first order; then the
    LayerNorm's own K u term and half an output ulp.  Heights below the 3-row halo, not multiples of the 4-row group, and
    with a partial last block; a common bias offset for half of them."""
    for i, H in enumerate((1, 2, 3, 4, 5, 13, 16, 17, 31)):
        B = 2
        offset = 6.0 if i % 2 else 0.0
        x, w49, bias, lw, lb = _dw_random(B, H, W, C, dtype, offset, seed=C * 100 + H)
        y = _dwconv(x, w49, bias, lw, lb).double()
        v = _conv64(x, w49, bias)
        dv = 50 * U24 * (_conv64(x.abs(), w49.abs(), None) + bias.double().abs())
        _, d, rstd = _ln64(v)
        ref = d * rstd * lw.double() + lb.double()
        bound = _dw_bound(v, rstd, lw, lb, C, dv, shifted=dtype == BF16)
        _check(f"dwconv_ln random {dtype} C={C} W={W} H={H} offset={offset}", y, ref, bound, dtype == BF16,
               FRAC_DW_LIMIT if dtype == BF16 else None)


@pytest.mark.parametrize("dtype", [BF16, torch.float32])
@pytest.mark.parametrize("C,W,H", [(96, 56, 9), (192, 28, 6), (768, 7, 17)])
def test_dwconv_ln_ragged_equals_clip_alone(C, W, H, dtype):
    """acx_dwconv_ln_ragged with clip b at h_b rows (1, H and heights between) in one launch: the input rows at or past
    h_b hold NaN and are never read, and the output rows below h_b equal acx_dwconv_ln of that clip alone at height h_b,
    bit for bit.  (The rows past h_b carry no promise and are not checked.)"""
    hs = [H, 1, max(2, H // 2), H - 1, 3]
    B = len(hs)
    x, w49, bias, lw, lb = _dw_random(B, H, W, C, dtype, 4.0, seed=C + H)
    for b, h in enumerate(hs):
        x[b, h:] = NAN
    valid = torch.tensor(hs, device=DEV, dtype=torch.int32)
    y = _dwconv(x, w49, bias, lw, lb, valid)
    for b, h in enumerate(hs):
        alone = _dwconv(x[b:b + 1, :h].contiguous(), w49, bias, lw, lb)
        assert torch.isfinite(alone.float()).all(), (C, h)
        assert torch.equal(y[b, :h], alone[0]), (C, dtype, b, h)


# ======================================================================================================================
# C.  ln_patchify / ln_patchify_gp
# ======================================================================================================================
def _patch_ref(x, lw, lb):
    """fp64 LayerNorm of every pixel of x (B, H, W, C) gathered to the patch matrix (B Ho Wo, 4C), k = (dy 2 + dx) C + c,
    with the per-element fp32 magnitudes (|x| + mean|x|) rstd |ln_w| and |ln_b| alongside, and the statistics."""
    B, H, W, C = x.shape
    Ho, Wo = H // 2, W // 2
    v = x[:, :2 * Ho, :2 * Wo].double()
    mean, d, rstd = _ln64(v)
    y = d * rstd * lw.double() + lb.double()
    mag = (v.abs() + v.abs().mean(-1, keepdim=True)) * rstd * lw.double().abs()

    def gather(t):
        return t.expand(B, 2 * Ho, 2 * Wo, t.shape[-1]).reshape(B, Ho, 2, Wo, 2, -1).permute(0, 1, 3, 2, 4, 5) \
            .reshape(B * Ho * Wo, -1)

    return gather(y), gather(mag), gather(mean), gather(rstd), gather(v)


def _lnp_K(C):
    """ln_patchify: 24 channels summed in sequence per lane, log2(C / 24) shuffle levels (depth <= 28) for the sum and for
    the squared deviations; + the division by C, the deviation, sqrtf, the reciprocal and the affine step."""
    return 24 + int(math.log2(C // 24)) + 8


# (C, W, H, B): stage widths, odd H (the dropped last row holds NaN) and even H
LNP_SHAPES = [(96, 56, 7, 2), (96, 56, 10, 1), (192, 28, 9, 2), (384, 14, 13, 2), (384, 14, 6, 3)]


@pytest.mark.parametrize("C,W,H,B", LNP_SHAPES)
def test_ln_patchify_readout(C, W, H, B):
    """acx_ln_patchify (bf16, fp32) and acx_ln_patchify_gp: every entry of the patch matrix against the fp64 LayerNorm at
    its patch position, within half an output ulp (bf16) + K u (|x| + mean|x|) rstd |ln_w| + 2 u |ln_b|, on closed-form
    rows, full-mantissa offset rows (mean / sigma 64 .. 400) and rows with u^2 near eps.  The dropped odd row and the
    planar padding rows hold NaN."""
    lw, lb = _affine(C, seed=3 * C + H)
    P = B * H * W
    Mo = B * (H // 2) * (W // 2)
    for dtype in (BF16, torch.float32):
        x = _ln_rows(P, C, dtype, seed=C + H).view(B, H, W, C)
        if H % 2:
            x[:, H - 1] = NAN
        ref, mag, _, _, _ = _patch_ref(x, lw, lb)
        bound = _lnp_K(C) * U24 * mag + 2 * U24 * lb.double().abs().repeat(4)
        a = torch.full((Mo + 3, 4 * C), NAN, device=DEV, dtype=dtype)
        N.call("acx_ln_patchify", x.data_ptr(), lw.data_ptr(), lb.data_ptr(), a.data_ptr(), B, H, W, C, _adt(dtype), _st())
        torch.cuda.synchronize()
        assert torch.isnan(a[Mo:].float()).all(), "wrote past the patch matrix"
        _check(f"ln_patchify {dtype} C={C} H={H}", a[:Mo].double(), ref, bound, dtype == BF16)
        if dtype == BF16:
            xg = _to_gp_nan(x.view(P, C))
            ag = torch.full((Mo, 4 * C), NAN, device=DEV, dtype=BF16)
            N.call("acx_ln_patchify_gp", xg.data_ptr(), lw.data_ptr(), lb.data_ptr(), ag.data_ptr(), B, H, W, C, _st())
            _check(f"ln_patchify_gp C={C} H={H}", ag.double(), ref, bound, True)
            assert torch.equal(ag, a[:Mo]), "planar and row-major forms differ"


# ======================================================================================================================
# D.  ds_fused (acx_downsample_fused_gp)
# ======================================================================================================================
def _ds_shapes(C):
    """(W, H, B): one shape with >= 3 tiles per persistent CTA (the grid is min(tiles, 148 SMs); tiles >= 3 x 148, a partial
    last tile, odd H), and one with fewer tiles than SMs (odd H)."""
    return {96: [(56, 511, 8), (56, 13, 1)], 192: [(28, 1017, 8), (28, 7, 2)], 384: [(14, 2031, 4), (14, 9, 3)]}[C]


def _ds(xg, lw, lb, wf, bias, B, H, W, C, out_gp):
    """acx_downsample_fused_gp -> (Mo, 2C) row-major; the row-major form must leave the NaN rows past Mo alone."""
    Mo = B * (H // 2) * (W // 2)
    if out_gp:
        Mop = (Mo + 127) // 128 * 128
        o = torch.full((2 * C // 8, Mop, 8), NAN, device=DEV, dtype=BF16)
        N.call("acx_downsample_fused_gp", xg.data_ptr(), lw.data_ptr(), lb.data_ptr(), wf.data_ptr(), bias.data_ptr(),
               o.data_ptr(), B, H, W, C, 1, _st())
        return o[:, :Mo].permute(1, 0, 2).reshape(Mo, 2 * C)     # planar padding rows are documented as written
    o = torch.full((Mo + 5, 2 * C), NAN, device=DEV, dtype=BF16)
    N.call("acx_downsample_fused_gp", xg.data_ptr(), lw.data_ptr(), lb.data_ptr(), wf.data_ptr(), bias.data_ptr(),
           o.data_ptr(), B, H, W, C, 0, _st())
    torch.cuda.synchronize()
    assert torch.isnan(o[Mo:].float()).all(), "wrote past the last output row"
    return o[:Mo]


def _ds_input(B, H, W, C, x):
    """x (B, H, W, C) bf16 -> group-planar with NaN in the planar padding rows and in the dropped odd row."""
    x = x.clone()
    if H % 2:
        x[:, H - 1] = NAN
    return x, _to_gp_nan(x.view(B * H * W, C))


def _ds_operand_bound(C, v, mean, rstd, lw, lb, a):
    """fp32 error of the A operand before its bf16 rounding.  Statistics: two lanes per pixel each sum C/2 shifted values
    x - x0 (x0 the pixel's first channel) in sequence, then one add: depth D = C/2 + 2 on the mean of the shifted values
    and on their second moment E2; var = E2 - md^2 loses D u E2 / var relative.  Operand ((x - mean) rstd) ln_w + ln_b."""
    D = C / 2 + 2
    x0 = v[..., :1]
    E2 = ((v - x0) ** 2).mean(-1, keepdim=True)
    var_eps = 1.0 / rstd ** 2
    mean_err = D * U24 * (v - x0).abs().mean(-1, keepdim=True) + U24 * mean.abs()
    rstd_rel = 0.5 * (D * U24 * E2 / var_eps + 2 * U24) + 5 * U24
    return lw.double().abs() * rstd * ((v - mean).abs() * (rstd_rel + 3 * U24) + mean_err) + \
        2 * U24 * (a.abs() + lb.double().abs())


def _ds_operand_ref(x, lw, lb, C):
    """exact operand (Mo, 4C) in the natural order k = (dy 2 + dx) C + c, and its fp32 error bound."""
    B, H, W, _ = x.shape
    Ho, Wo = H // 2, W // 2
    v = x[:, :2 * Ho, :2 * Wo].double()
    mean, d, rstd = _ln64(v)
    a = d * rstd * lw.double() + lb.double()
    da = _ds_operand_bound(C, v, mean, rstd, lw, lb, a)
    del v, d

    def gather(t):
        return t.reshape(B, Ho, 2, Wo, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(B * Ho * Wo, 4 * C)

    return gather(a), gather(da)


def _natural_weight(w4):
    """(2C, C, 2, 2) conv weight -> (2C, 4C) in the natural patch order k = (dy 2 + dx) C + c."""
    return w4.permute(0, 2, 3, 1).reshape(w4.shape[0], -1)


@pytest.mark.parametrize("C", [96, 192, 384])
def test_ds_fused_operand_readout(C):
    """The bf16 A operand of acx_downsample_fused_gp, read out exactly: selector conv weights (output column n of launch j
    reads natural K entry 2 C j + n with weight 1, bias 0, packed by engine.pack_downsample_weight) turn the fp32
    accumulation into a copy, so two launches read all 4C entries.  Against the fp64 LayerNorm within half an ulp + the
    fp32 bound of the shifted single-pass statistics, on closed-form rows, full-mantissa offset rows, u^2 ~ eps rows and
    rows whose first channel is far from the mean; with >= 3 tiles per CTA and with fewer tiles than SMs, odd H, both
    output layouts."""
    from audioset_convnext_inf_b200.engine import pack_downsample_weight
    lw, lb = _affine(C, seed=7 * C)
    zero = torch.zeros(2 * C, device=DEV)
    sel = []
    for j in range(2):
        w4 = torch.zeros(2 * C, C, 2, 2)
        k = 2 * C * j + torch.arange(2 * C)
        q, c = k // C, k % C
        w4[torch.arange(2 * C), c, q // 2, q % 2] = 1.0
        assert torch.equal(_natural_weight(w4)[:, 2 * C * j:2 * C * (j + 1)], torch.eye(2 * C))
        sel.append(pack_downsample_weight(w4).to(BF16).contiguous().to(DEV))
    for W, H, B in _ds_shapes(C):
        Mo = B * (H // 2) * (W // 2)
        tiles = (Mo + 127) // 128 * (1 if C < 384 else 2)
        x, xg = _ds_input(B, H, W, C, _ln_rows(B * H * W, C, BF16, seed=C + H, far_first=True).view(B, H, W, C))
        ref, da = _ds_operand_ref(x, lw, lb, C)
        for out_gp in (0, 1):
            got = torch.cat([_ds(xg, lw, lb, s, zero, B, H, W, C, out_gp) for s in sel], 1).double()
            _check(f"ds_fused operand C={C} H={H} B={B} tiles={tiles} out_gp={out_gp}", got, ref, da, True)


# Fraction of ds_fused outputs that differ from the round-to-nearest of the fp64 emulation (random operands, common row
# offsets).  Measured on one NVIDIA B200 (1000 W power limit): 0.104 / 0.257 / 0.720 % at C = 96 / 192 / 384, both layouts.
FRAC_DS_LIMIT = 0.015


@pytest.mark.parametrize("C", [96, 192, 384])
def test_ds_fused_emulated_rounding(C):
    """acx_downsample_fused_gp on random operands with common row offsets against an fp64 emulation: the operand
    ((x - mean) rstd) ln_w + ln_b rounded to bf16 (entries within their fp32 slack of a rounding boundary flagged as
    uncertain), the fp32 accumulation over K = 4C, + bias, one bf16 rounding.  Per element
    |got - emul| <= 0.5 ulp + sum over uncertain k of ulp(a_k) |w_nk| + 2 K u sum |a_k w_nk| + u |acc|, and in aggregate the
    fraction of outputs != RN(emul) stays below FRAC_DS_LIMIT.  Multi-tile shapes, both output layouts."""
    from audioset_convnext_inf_b200.engine import pack_downsample_weight
    W, H, B = _ds_shapes(C)[0]
    g = torch.Generator().manual_seed(C)
    P = B * H * W
    x = (torch.randn(P, C, generator=g) * (1.0 + 3.0 * torch.rand(P, 1, generator=g)) +
         3.0 * torch.randn(P, 1, generator=g)).to(BF16).view(B, H, W, C).to(DEV)
    w4 = (torch.randn(2 * C, C, 2, 2, generator=g) / (4 * C) ** 0.5).to(BF16)
    bias = (torch.randn(2 * C, generator=g) * 0.1).to(DEV)
    lw, lb = _affine(C, seed=11 * C)
    wf = pack_downsample_weight(w4).contiguous().to(DEV)
    wn = _natural_weight(w4).double().to(DEV)
    x, xg = _ds_input(B, H, W, C, x)
    a, da = _ds_operand_ref(x, lw, lb, C)
    aq = _rn(a)
    unc = ((a - aq).abs() + da >= 0.5 * _ulp((a.abs() - da).clamp_min(0.0))).double()
    del a
    acc = aq @ wn.t()
    emul = acc + bias.double()
    d = (unc * _ulp(aq)) @ wn.abs().t() + 2 * 4 * C * U24 * (aq.abs() @ wn.abs().t()) + U24 * emul.abs()
    print(f"  ds_fused C={C}: uncertain operand entries {100 * unc.mean().item():.3f} %")
    del unc, aq
    for out_gp in (0, 1):
        got = _ds(xg, lw, lb, wf, bias, B, H, W, C, out_gp).double()
        _check(f"ds_fused random C={C} out_gp={out_gp}", got, emul, d, True, FRAC_DS_LIMIT)
