"""GPU (B200): rounding-level tests of the bf16 tensor-core kernels and of the stem / head / front-end pieces.

The bit-identity tests of ragged batches, windows, streams, SED and search all reduce to "equal to the clip run alone", so
the arithmetic of the exact-length path is what everything rests on.  These tests bound each kernel by its own documented
arithmetic instead of by a loose multiple of the output magnitude:

* A  GELU readouts: W1 rows are scaled unit vectors and b1 = 0, so every pre-activation is ONE bf16 x bf16 product (exact
     in fp32) and the output is the kernel's GELU rounded once to bf16 -- every bf16 value in [-12, 12] times four scales,
     the clamp region, +-0 and tiny magnitudes, on every GELU-bearing kernel.
* B  LayerNorm readouts: rows +-u around a mean, whose statistics are exact in the kernels' shifted single-pass arithmetic,
     with u^2 comparable to eps and with large common offsets; and full-mantissa rows with mean / sigma up to 400, on
     which a variance without the shift cancels.
* C  emulated-rounding bounds on random operands: fp64 emulation of the documented rounding points, per element and in
     aggregate (the fraction of outputs that differ from the round-to-nearest of the emulation).
* D  stem at every frame count mod 4 (dense, planar and ragged forms), head at h3 = 1, power -> mel -> dB -> bn0, and the
     model end to end against the fp64 oracle at the clip lengths whose shapes the golden tests never reach.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

from audioset_convnext_inf_b200 import _native as N          # noqa: E402
from oracle import convnext_oracle as O                       # noqa: E402
from oracle import weights                                    # noqa: E402

DEV = "cuda:0"
F64 = torch.float64

# Largest |tensor-core GELU - exact erf GELU| (common.cuh, "max |err|"), fp32 arithmetic and tanh.approx.f32 included.
# Measured through the readouts below on one NVIDIA B200 (1000 W power limit): at most 2.50e-5 beyond half an output ulp,
# at x = -3.07, the same on every GELU-bearing kernel; below x = -3 at most 3.3e-5 in all (half an ulp included).
GELU_E = 2.6e-5
U24 = 2.0 ** -24                       # fp32 unit roundoff
SCALES = (1.0, 0.75, 1.25, -0.5625)    # bf16-exact multipliers of the pre-activation sweep (one per 128-column group of C)
# golden tolerances of tests/test_gpu_model.py (TOL): logits, scene and frame against the oracle
TOL = {"fp32": dict(logits=1e-4 * 5, scene=5e-4, frame=2e-3), "bf16": dict(logits=2e-2 * 3, scene=0.12, frame=0.6)}


def _st():
    return torch.cuda.current_stream().cuda_stream


# ---- fp64 models of the roundings -----------------------------------------------------------------------------------
def _ulp(v):
    """bf16 spacing at |v| (normal range)."""
    return torch.exp2(torch.floor(torch.log2(v.abs().clamp_min(2.0 ** -126))) - 7)


def _rn(v):
    """fp64 -> nearest bf16 value (ties to even), without a detour through fp32."""
    q = _ulp(v)
    return torch.round(v / q) * q


def _gelu(x):
    """exact erf GELU in fp64, accurate in the negative tail (erfc, not 1 + erf)."""
    return 0.5 * x * torch.special.erfc(-x / math.sqrt(2.0))


def _to_gp(t):
    """(M, C) -> group-planar [C/8][Mp][8], Mp = M rounded up to 128."""
    M, C = t.shape
    Mp = (M + 127) // 128 * 128
    out = torch.zeros(C // 8, Mp, 8, device=t.device, dtype=t.dtype)
    out[:, :M] = t.view(M, C // 8, 8).permute(1, 0, 2)
    return out


def _from_gp(t, M, C):
    return t.view(C // 8, -1, 8)[:, :M].permute(1, 0, 2).reshape(M, C).contiguous()


# ---- the kernels under test -------------------------------------------------------------------------------------------
def _mlp(kind, y, x, w1, b1, w2, b2, gamma, ln_w=None, ln_b=None, ln_s=None):
    """One fused-MLP launch; y / x (M, C) bf16 row-major in, the updated x (M, C) row-major out."""
    M, C = x.shape
    st = _st()
    tail = (w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(), gamma.data_ptr(), M, C, st)
    if kind == "rm":
        out = x.clone()
        N.call("acx_mlp_fused", y.data_ptr(), out.data_ptr(), *tail)
        return out
    if kind == "ln":
        out = x.clone()
        N.call("acx_mlp_fused_ln", y.data_ptr(), out.data_ptr(), ln_w.data_ptr(), ln_b.data_ptr(), *tail)
        return out
    yg, xg = _to_gp(y), _to_gp(x)
    p = lambda t: t.data_ptr() if t is not None else 0           # noqa: E731
    N.call("acx_mlp_fused_gp", yg.data_ptr(), xg.data_ptr(), p(ln_w), p(ln_b), p(ln_s), *tail)
    return _from_gp(xg, M, C)


def _gemm(A, W, epi, bias, gamma=None, resid=None):
    M, K = A.shape
    Nn = W.shape[0]
    out = torch.full((M, Nn), float("nan"), device=DEV, dtype=torch.bfloat16)
    N.call("acx_gemm_bf16", A.data_ptr(), W.data_ptr(), out.data_ptr(), M, Nn, K, epi, bias.data_ptr(),
           gamma.data_ptr() if gamma is not None else 0, resid.data_ptr() if resid is not None else 0, _st())
    return out


def _pw1_gp(v, w1f, b1f, s1, stats):
    M, K = v.shape
    hid = torch.full((M, w1f.shape[0]), float("nan"), device=DEV, dtype=torch.bfloat16)
    N.call("acx_gemm_bf16_pw1_gp", _to_gp(v).data_ptr(), w1f.data_ptr(), hid.data_ptr(), M, w1f.shape[0], K, b1f.data_ptr(),
           stats.data_ptr(), s1.data_ptr(), _st())
    return hid


def _row_stats(v):
    M, C = v.shape
    stats = torch.full((M, 2), float("nan"), device=DEV)
    N.call("acx_gp_row_stats", _to_gp(v).data_ptr(), stats.data_ptr(), M, C, _st())
    return stats


# ======================================================================================================================
# A. GELU readouts through designed operands
# ======================================================================================================================
def _sweep_values():
    """Every bf16 value in [-12, 12] with |x| >= 2^-100 (products with the scales stay fp32-normal), +-0, tiny
    magnitudes and the clamp region |x| > sqrt(50) up to 1e30."""
    b = torch.arange(65536, dtype=torch.int32).to(torch.int16).view(torch.bfloat16).to(F64)
    b = b[torch.isfinite(b) & (b.abs() <= 12) & ((b.abs() >= 2.0 ** -100) | (b == 0))]
    extra = torch.tensor([0.0, -0.0, 2.0 ** -100, -(2.0 ** -100), 2.0 ** -60, -(2.0 ** -60), 16.0, -16.0, 100.0, -100.0,
                          1024.0, -1024.0, 65536.0, -65536.0, 1e30, -1e30], dtype=F64)
    return torch.cat([b, _rn(extra)])


def _readout_operands(C, M, seed):
    """y (M, C): the sweep, repeated and shuffled; W1 row j = SCALES[j // C] e_(j mod C); b1 = 0."""
    vals = _sweep_values()
    g = torch.Generator().manual_seed(seed)
    n = M * C
    y = vals[torch.randint(0, vals.numel(), (n,), generator=g)]
    y[: vals.numel()] = vals                                      # every value at least once
    y = y[torch.randperm(n, generator=g)].view(M, C)
    w1 = torch.zeros(4 * C, C, dtype=F64)
    for j in range(4 * C):
        w1[j, j % C] = SCALES[j // C]
    pre = torch.cat([y * s for s in SCALES], 1)                  # (M, 4C): pre[m, j] = y[m, j % C] * SCALES[j // C]
    return y.to(torch.bfloat16).to(DEV), w1.to(torch.bfloat16).to(DEV), pre.to(DEV)


def _check_gelu_readout(tag, got, pre):
    """got: the kernel's bf16 GELU of the exact pre-activations `pre` (both fp64 on the device)."""
    assert torch.isfinite(got).all(), f"{tag}: unwritten or non-finite outputs"
    ref = _gelu(pre)
    err = (got - ref).abs()
    excess = err - 0.5 * _ulp(got)
    i = int(excess.argmax())
    # one bf16 ulp of bf16(gelu) wherever the GELU's own error E is below ~half an ulp (x >= -3: |gelu| >= 4e-3)
    rr = _rn(ref)
    ulps = (got - rr).abs() / _ulp(rr)
    body = pre >= -3.0
    tail = (pre < -3.0) & (pre > -12.0)
    print(f"  {tag}: max |got - gelu| beyond half an ulp {excess.max().item():.3e} at x = {pre.flatten()[i].item():.6g} "
          f"(gelu {ref.flatten()[i].item():.4e}, got {got.flatten()[i].item():.4e}); max |err| in x<-3 "
          f"{err[tail].max().item():.3e}; max ulps from bf16(gelu) for x>=-3: {ulps[body].max().item():.0f}")
    assert (ulps[body] <= 1).all(), (tag, ulps[body].max().item())
    assert (err <= 0.5 * _ulp(got) + GELU_E).all(), (tag, excess.max().item(), pre.flatten()[i].item())
    # the clamp region: gelu(x) = x above sqrt(50), 0 (either sign) below -sqrt(50)
    big = pre > 50 ** 0.5
    assert torch.equal(got[big], _rn(pre[big]))
    assert (got[pre < -(50 ** 0.5)].abs() <= GELU_E).all()
    zero = pre == 0
    assert (got[zero] == 0).all()


@pytest.mark.parametrize("C", [96, 192])
def test_gelu_readout_gemm_and_fused_mlps(C):
    """The GELU of acx_gemm_bf16 (EPI_BIAS_GELU), acx_gemm_bf16_pw1_gp (stats (1, 0): no LayerNorm), acx_mlp_fused and
    acx_mlp_fused_gp, read out directly.  For the fused MLPs W2 selects hidden column q C + c for output channel c with
    weight 1, gamma = 1, b2 = 0, x = 0: the output is bf16(2 gelu) / 2 exactly, and four selections read all 4C hidden
    columns (every 128-column D1 chunk).  M gives every persistent CTA more than two row tiles."""
    M = 128 * 148 * 2 + 77
    y, w1, pre = _readout_operands(C, M, seed=C)
    z4, zc = torch.zeros(4 * C, device=DEV), torch.zeros(C, device=DEV)
    ones = torch.ones(C, device=DEV)
    _check_gelu_readout(f"gemm_bf16 GELU C={C}", _gemm(y, w1, N.EPI_BIAS_GELU, z4).double(), pre)
    if C % 64 == 0:                                               # a planar A operand needs K % 64 == 0
        stats = torch.tensor([1.0, 0.0], device=DEV).expand(M, 2).contiguous()
        _check_gelu_readout(f"gemm_bf16_pw1_gp C={C}", _pw1_gp(y, w1, z4, z4, stats).double(), pre)
    x0 = torch.zeros(M, C, device=DEV, dtype=torch.bfloat16)
    for kind in ("rm", "gp"):
        got = torch.empty(M, 4 * C, device=DEV, dtype=F64)
        for q in range(4):
            w2 = torch.zeros(C, 4 * C, device=DEV)
            w2[torch.arange(C), q * C + torch.arange(C)] = 1.0
            out = _mlp(kind, y, x0, w1, z4, w2.to(torch.bfloat16), zc, ones)
            got[:, q * C:(q + 1) * C] = out.double()
        _check_gelu_readout(f"mlp_fused[{kind}] C={C}", got, pre)


# ======================================================================================================================
# B. LayerNorm readouts
# ======================================================================================================================
# (mean, u): rows mean +- u alternating by channel, every value bf16-exact, so every partial sum of the statistics is exact in
# fp32 and rstd / mean are known in closed form.  u^2 comparable to eps = 1e-6 (a wrong eps moves rstd by tens of percent).
LN_ROWS = [(0.0, 2.0 ** -10), (0.0, 2.0 ** -11), (0.0, 2.0 ** -9), (0.0, 2.0 ** -12), (0.0, 0.5), (64.0, 0.5),
           (128.0, 1.0), (-96.0, 0.5), (8.0, 2.0 ** -4), (1.0, 2.0 ** -7), (-2.0, 2.0 ** -6), (16.0, 2.0 ** -3)]
# (mean, sigma): bf16 rows mean + sigma N(0, 1), mean / sigma from 64 to 400, whose sums round in fp32.  There a single-pass
# variance without the shift (E[v^2] - mean^2) loses 1e-3 .. 1e-2 of rstd; shifted by the row's first channel, ~1e-6.
LN_OFFSET_ROWS = [(16.0, 0.25), (64.0, 0.5), (128.0, 1.0), (100.0, 0.25)]


def _ln_operands(C, M):
    """Rows LN_ROWS then LN_OFFSET_ROWS, cycling.  Returns v (bf16), mean, rstd, v - mean (fp64), and per row the fp32 slack
    of the statistics beyond exact sums -- relative on rstd, absolute on the mean -- which is zero for the closed-form
    rows.  On the offset rows any order of summing C terms errs by at most (C - 1) u sum |terms|: a variance shifted by
    the first channel v0 by C u E[(v - v0)^2] / (var + eps) relative, the mean by C u E|v - v0|."""
    nr = len(LN_ROWS) + len(LN_OFFSET_ROWS)
    fam = torch.arange(M) % nr
    rows = LN_ROWS + LN_OFFSET_ROWS
    mu = torch.tensor([r[0] for r in rows], dtype=F64)[fam]
    u = torch.tensor([r[1] for r in rows], dtype=F64)[fam]
    sign = 1.0 - 2.0 * (torch.arange(C) % 2).to(F64)
    z = torch.randn(M, C, generator=torch.Generator().manual_seed(C + M), dtype=F64)
    closed = fam < len(LN_ROWS)
    v = torch.where(closed[:, None], mu[:, None] + u[:, None] * sign[None, :], mu[:, None] + u[:, None] * z)
    v = v.to(torch.bfloat16).double()
    assert torch.equal(v[closed], mu[closed, None] + u[closed, None] * sign[None, :])
    mean = v.mean(1)
    dev = v - mean[:, None]
    var = (dev * dev).mean(1)
    rstd = 1.0 / torch.sqrt(var + 1e-6)
    assert torch.equal(mean[closed], mu[closed]) and torch.equal(var[closed], u[closed] ** 2)
    sh = v - v[:, :1]
    rel = torch.where(closed, 0.0, 0.5 * C * U24 * (sh * sh).mean(1) / (var + 1e-6))
    mean_err = torch.where(closed, 0.0, C * U24 * sh.abs().mean(1))
    return (v.to(torch.bfloat16).to(DEV), mean.to(DEV), rstd.to(DEV), dev.to(DEV),
            (rel.to(DEV)[:, None], mean_err.to(DEV)[:, None]))


def test_layernorm_statistics_readout():
    """acx_gp_row_stats and acx_layernorm_rows on rows with closed-form statistics: rstd = 1 / sqrt(u^2 + 1e-6) to fp32
    accuracy, -mean rstd likewise, and LN(v) within one bf16 rounding of its fp64 value; on the full-mantissa offset rows
    the same plus the rounding of the (shifted) sums."""
    for C in (96, 192, 384):
        M = 128 * 3 + 5
        v, mu, rstd, dev, (rel, mean_err) = _ln_operands(C, M)
        rel, mean_err = rel[:, 0], mean_err[:, 0]
        stats = _row_stats(v).double()
        assert ((stats[:, 0] - rstd).abs() <= (4 * U24 + rel) * rstd).all(), ((stats[:, 0] / rstd - 1).abs().max().item())
        assert ((stats[:, 1] + mu * rstd).abs() <= (4 * U24 + rel) * (mu * rstd).abs() + mean_err * rstd + 1e-30).all(), \
            ((stats[:, 1] + mu * rstd).abs() - (4 * U24 + rel) * (mu * rstd).abs() - mean_err * rstd).max().item()
        g = torch.Generator().manual_seed(C)
        lw = (torch.rand(C, generator=g) * 0.4 + 0.8).to(DEV)
        lb = (torch.randn(C, generator=g) * 0.1).to(DEV)
        y = torch.full_like(v, float("nan"))
        N.call("acx_layernorm_rows", v.data_ptr(), lw.data_ptr(), lb.data_ptr(), y.data_ptr(), M, C, _st())
        ref = dev * rstd[:, None] * lw.double() + lb.double()
        # out = v (rstd w) + (b - mean rstd w) in fp32: the two terms cancel for rows with a large common offset
        slack = (((v.double().abs() + mu.abs()[:, None]) * rstd[:, None] * lw.double()).abs() + lb.double().abs()) * 8 * U24
        slack = slack + (rel[:, None] * dev.abs() + mean_err[:, None]) * rstd[:, None] * lw.double().abs()
        yd = y.double()
        assert ((yd - ref).abs() <= 0.5 * _ulp(yd) + slack).all(), ((yd - ref).abs() / _ulp(yd)).max().item()


@pytest.mark.parametrize("C", [96, 192])
def test_layernorm_readout_through_the_gelu(C):
    """The LayerNorm of the fused MLPs (in shared memory: acx_mlp_fused_ln, acx_mlp_fused_gp with ln_w / ln_b; folded:
    acx_mlp_fused_gp with ln_s) and of stage 2 (acx_gp_row_stats + acx_gemm_bf16_pw1_gp), read through a selector W1
    (scales s_j, b1 = 0) and a selector W2: pre = rstd (v - mean) s_j in closed form.  Bound: the fp32 error of the
    statistics and of the fold's cancellation, one bf16 rounding of the normalised operand (in-smem form), the GELU's E,
    and the output rounding."""
    M = 128 * 150 + 77
    v, mu, rstd, dev, (rel, mean_err) = _ln_operands(C, M)
    w1 = torch.zeros(4 * C, C)
    for j in range(4 * C):
        w1[j, j % C] = SCALES[j // C]
    w1 = w1.to(torch.bfloat16).to(DEV)
    s1 = w1.float().sum(1)
    sc = torch.tensor(SCALES, dtype=F64, device=DEV).repeat_interleave(C)
    yn = dev * rstd[:, None]                                      # LN(v) with ln_w = 1, ln_b = 0, fp64
    pre = yn.repeat(1, 4) * sc                                    # (M, 4C)
    z4, zc, ones = torch.zeros(4 * C, device=DEV), torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    x0 = torch.zeros(M, C, device=DEV, dtype=torch.bfloat16)

    def read(kind, **ln):
        got = torch.empty(M, 4 * C, device=DEV, dtype=F64)
        for q in range(4):
            w2 = torch.zeros(C, 4 * C, device=DEV)
            w2[torch.arange(C), q * C + torch.arange(C)] = 1.0
            got[:, q * C:(q + 1) * C] = _mlp(kind, v, x0, w1, z4, w2.to(torch.bfloat16), zc, ones, **ln).double()
        return got

    # in-smem LayerNorm: the normalised operand is rounded to bf16 before GEMM1
    d_smem = (0.5 * _ulp(yn) + yn.abs() * 8 * U24).repeat(1, 4) * sc.abs()
    # folded: pre = rstd G + (-mean rstd) s + b1 in fp32, G = v_k s_j exact; the two terms cancel
    big = (mu.abs() + dev.abs().amax(1))[:, None] * rstd[:, None] * sc.abs()
    d_fold = big * 8 * U24
    # offset rows: the rounding of the statistics' sums, the same in every form
    d_stats = ((rel * dev.abs() + mean_err) * rstd[:, None]).repeat(1, 4) * sc.abs()
    d_smem, d_fold = d_smem + d_stats, d_fold + d_stats
    lw, lb = ones, zc
    cases = [("mlp_fused_ln", read("ln", ln_w=lw, ln_b=lb), d_smem),
             ("mlp_fused_gp ln_w/ln_b", read("gp", ln_w=lw, ln_b=lb), d_smem),
             ("mlp_fused_gp folded", read("gp", ln_s=s1), d_fold),
             ] + ([("gp_row_stats + pw1_gp", _pw1_gp(v, w1, z4, s1, _row_stats(v)).double(), d_fold)] if C % 64 == 0 else [])
    for tag, got, d in cases:
        assert torch.isfinite(got).all(), tag
        err = (got - _gelu(pre)).abs()
        bound = 0.5 * _ulp(got) + GELU_E + 1.13 * d
        print(f"  LN readout {tag} C={C}: max (|err| - bound) {(err - bound).max().item():.3e}")
        assert (err <= bound).all(), (tag, (err - bound).max().item())


# ======================================================================================================================
# C. Emulated-rounding bounds on random operands
# ======================================================================================================================
def _rand_mlp(C, M, seed, offset=0.0):
    g = torch.Generator().manual_seed(seed)
    y = (torch.randn(M, C, generator=g) * (1.0 + offset * torch.rand(M, 1, generator=g)) +
         offset * torch.randn(M, 1, generator=g)).to(torch.bfloat16)
    x = torch.randn(M, C, generator=g).to(torch.bfloat16)
    w1 = torch.randn(4 * C, C, generator=g) / C ** 0.5
    w2 = (torch.randn(C, 4 * C, generator=g) / (4 * C) ** 0.5).to(torch.bfloat16)
    b1 = torch.randn(4 * C, generator=g) * 0.1
    b2 = torch.randn(C, generator=g) * 0.3
    gamma = torch.rand(C, generator=g) * 0.5 + 0.1
    lw = torch.rand(C, generator=g) * 0.4 + 0.8
    lb = torch.randn(C, generator=g) * 0.05
    return [t.to(DEV) for t in (y, x, w1, w2, b1, b2, gamma, lw, lb)]


def _hidden_emulation(pre, d_pre):
    """The bf16 hidden 2 gelu(pre) of the fused MLP: its round-to-nearest value, and per column whether the kernel's value
    (within 2 (E + 1.13 d_pre) of 2 gelu(pre)) may round to the other neighbour."""
    v = 2.0 * _gelu(pre)
    h = _rn(v)
    unc = 2.0 * (GELU_E + 1.13 * d_pre)
    uncertain = (v - h).abs() + unc >= 0.5 * _ulp((v.abs() - unc).clamp_min(0.0))
    return h, uncertain


def _check_fused_emulation(tag, got, x, h, uncertain, w2, b2, gamma, limit):
    """Per element  |got - emul| <= (0.5 + MLP_EXTRA_ULP) ulp(got) + sum_j |c_kj| ulp(h_j) over uncertain j + fp32 slack,
    c = 0.5 gamma W2;
    in aggregate the fraction of outputs != RN(emul) stays below `limit`."""
    w2d, gd = w2.double(), gamma.double()
    emul = x.double() + 0.5 * gd * (h @ w2d.t()) + gd * b2.double()
    unc = 0.5 * gd * ((uncertain.double() * _ulp(h)) @ w2d.abs().t())
    acc_abs = 0.5 * gd * (h.abs() @ w2d.abs().t())
    slack = 2 * w2.shape[1] * U24 * acc_abs + (x.double().abs() + (gd * b2.double()).abs() + acc_abs) * 3 * U24
    err = (got - emul).abs()
    excess = err - ((0.5 + MLP_EXTRA_ULP) * _ulp(got) + unc + slack)
    frac = (got != _rn(emul)).double().mean().item()
    bad = torch.nonzero(excess > 0)
    if bad.numel():
        print(f"  {tag}: {bad.shape[0]} elements over the bound; rows mod 128 {sorted(set((bad[:, 0] % 128).tolist()))[:16]}, "
              f"tiles {sorted(set((bad[:, 0] // 128).tolist()))[:16]}, channels {sorted(set(bad[:, 1].tolist()))[:16]}")
    print(f"  {tag}: max excess over the bound {excess.max().item():.3e}; outputs != RN(emulation): {100 * frac:.2f} % "
          f"(uncertain hidden columns {100 * uncertain.double().mean().item():.2f} %)")
    assert (excess <= 0).all(), (tag, excess.max().item())
    assert frac < limit, (tag, frac)
    return frac


# Fraction of outputs that differ from the round-to-nearest of the fp64 emulation.  Measured on one NVIDIA B200 (1000 W
# power limit): fused MLPs 2.1-3.6 %; GEMM with the GELU epilogue 1.8-1.9 %; bias, scale + residual, planar output and
# pw2 at most 0.08 %.  CPU emulation of the fused MLP gives ~3 % for the documented arithmetic, 9 % with the textbook
# tanh GELU, 29 % with the hidden tile rounded toward zero and 50 % with the output rounded toward zero.
FRAC_MLP_LIMIT = 0.06
FRAC_GELU_LIMIT = 0.04
FRAC_GEMM_LIMIT = 0.005
# Per-element slack of the fused MLPs beyond the emulated bound, in output ulps: on the B200 above, 5 of 3.6 M outputs of
# the C = 96 kernel exceeded the half-ulp bound, by at most 0.66 ulp.
MLP_EXTRA_ULP = 1.0


@pytest.mark.parametrize("C,M", [(96, 128 * 148 * 2 + 77), (192, 128 * 150 + 5)])
def test_fused_mlp_emulated_rounding(C, M):
    """acx_mlp_fused, acx_mlp_fused_ln, acx_mlp_fused_gp (plain, in-smem LayerNorm, folded LayerNorm) against the fp64
    emulation of their documented roundings on random operands."""
    from audioset_convnext_inf_b200.engine import fold_layernorm_into_pwconv1
    y, x, w1, w2, b1, b2, gamma, lw, lb = _rand_mlp(C, M, seed=C + M, offset=3.0)
    w1b = w1.to(torch.bfloat16)
    w1d = w1b.double()
    # plain: pre = y W1^T + b1, fp32 accumulation
    yd = y.double()
    pre = yd @ w1d.t() + b1.double()
    d_pre = 2 * C * U24 * (yd.abs() @ w1d.abs().t()) + pre.abs() * U24
    h, unc = _hidden_emulation(pre, d_pre)
    for kind in ("rm", "gp"):
        _check_fused_emulation(f"mlp_fused[{kind}] C={C}", _mlp(kind, y, x, w1b, b1, w2, b2, gamma).double(), x, h, unc, w2,
                               b2, gamma, FRAC_MLP_LIMIT)
    # in-smem LayerNorm: the operand LN(y) is rounded to bf16 first (an uncertain rounding widens d_pre)
    mean = yd.mean(1, keepdim=True)
    rstd = 1.0 / torch.sqrt(yd.var(1, unbiased=False, keepdim=True) + 1e-6)
    yn = (yd - mean) * rstd * lw.double() + lb.double()
    d_yn = (yd - mean).abs() * rstd * lw.double() * 16 * U24 * (1 + (mean.abs() / (yd - mean).abs().amax(1, keepdim=True)))
    yq = _rn(yn)
    y_unc = ((yn - yq).abs() + d_yn >= 0.5 * _ulp((yn.abs() - d_yn).clamp_min(0.0))).double()
    pre = yq @ w1d.t() + b1.double()
    d_pre = 2 * C * U24 * (yq.abs() @ w1d.abs().t()) + pre.abs() * U24 + (y_unc * _ulp(yq)) @ w1d.abs().t()
    h, unc = _hidden_emulation(pre, d_pre)
    for kind in ("ln", "gp"):
        got = _mlp(kind, y, x, w1b, b1, w2, b2, gamma, ln_w=lw, ln_b=lb).double()
        _check_fused_emulation(f"mlp_fused LN in smem [{kind}] C={C}", got, x, h, unc, w2, b2, gamma, FRAC_MLP_LIMIT)
    # folded LayerNorm: pre = rstd G + (-mean rstd) s + b1', G = y W1'^T with W1' = bf16(W1 ln_w)
    f = fold_layernorm_into_pwconv1(w1.cpu(), b1.cpu(), lw.cpu(), lb.cpu())
    w1f, s1, b1f = (f[k].to(DEV) for k in ("w1f", "s1", "b1f"))
    G = yd @ w1f.double().t()
    pre = rstd * G - mean * rstd * s1.double() + b1f.double()
    d_pre = (2 * C * U24 * (yd.abs() @ w1f.double().abs().t()) + G.abs() * 8 * U24) * rstd + \
        (mean * rstd * s1.double()).abs() * 8 * U24 + pre.abs() * U24
    h, unc = _hidden_emulation(pre, d_pre)
    got = _mlp("gp", y, x, w1f, b1f, w2, b2, gamma, ln_s=s1).double()
    _check_fused_emulation(f"mlp_fused folded LN C={C}", got, x, h, unc, w2, b2, gamma, FRAC_MLP_LIMIT)


def _check_gemm(tag, got, emul, d, limit):
    err = (got - emul).abs()
    excess = err - (0.5 * _ulp(got) + d)
    frac = (got != _rn(emul)).double().mean().item()
    print(f"  {tag}: max excess over the bound {excess.max().item():.3e}; outputs != RN(emulation): {100 * frac:.3f} %")
    assert torch.isfinite(got).all(), tag
    assert (excess <= 0).all(), (tag, excess.max().item())
    assert frac < limit, (tag, frac)


@pytest.mark.parametrize("M,Nn,K", [(14112, 384, 96), (3528, 768, 192), (882, 384, 1536), (128 * 700, 192, 192),
                                    (300, 192, 96)])
def test_gemm_emulated_rounding(M, Nn, K):
    """acx_gemm_bf16 (bias, bias + GELU, scale + residual) and acx_gemm_bf16_gp_out against fp64 with one bf16 rounding:
    |got - emul| <= 0.5 ulp(got) + the fp32 accumulation bound (+ E for the GELU)."""
    g = torch.Generator().manual_seed(M + Nn + K)
    A = torch.randn(M, K, generator=g).to(torch.bfloat16).to(DEV)
    W = (torch.randn(Nn, K, generator=g) / K ** 0.5).to(torch.bfloat16).to(DEV)
    bias = (torch.randn(Nn, generator=g) * 0.1).to(DEV)
    gamma = torch.rand(Nn, generator=g).to(DEV)
    resid = torch.randn(M, Nn, generator=g).to(torch.bfloat16).to(DEV)
    pre = A.double() @ W.double().t() + bias.double()
    d_pre = 2 * K * U24 * (A.double().abs() @ W.double().abs().t()) + pre.abs() * U24
    _check_gemm(f"gemm bias {M}x{Nn}x{K}", _gemm(A, W, N.EPI_BIAS, bias).double(), pre, d_pre, FRAC_GEMM_LIMIT)
    _check_gemm(f"gemm gelu {M}x{Nn}x{K}", _gemm(A, W, N.EPI_BIAS_GELU, bias).double(), _gelu(pre),
                GELU_E + 1.13 * d_pre + _gelu(pre).abs() * 2 * U24, FRAC_GELU_LIMIT)
    emul = resid.double() + gamma.double() * pre
    d = gamma.double() * d_pre + (resid.double().abs() + (gamma.double() * pre).abs()) * U24
    _check_gemm(f"gemm scale+resid {M}x{Nn}x{K}", _gemm(A, W, N.EPI_BIAS_SCALE_RESID, bias, gamma, resid).double(), emul, d,
                FRAC_GEMM_LIMIT)
    Mp = (M + 127) // 128 * 128
    og = torch.full((Nn // 8, Mp, 8), float("nan"), device=DEV, dtype=torch.bfloat16)
    N.call("acx_gemm_bf16_gp_out", A.data_ptr(), W.data_ptr(), og.data_ptr(), M, Nn, K, bias.data_ptr(), _st())
    _check_gemm(f"gemm gp_out {M}x{Nn}x{K}", _from_gp(og, M, Nn).double(), pre, d_pre, FRAC_GEMM_LIMIT)


@pytest.mark.parametrize("M", [64 * 63 * 14, 200])
def test_stage2_planar_gemms_emulated_rounding(M):
    """acx_gp_row_stats + acx_gemm_bf16_pw1_gp (LayerNorm folded into the GELU epilogue) and acx_gemm_bf16_pw2_gp on
    random operands with common row offsets, against fp64 emulations of their arithmetic."""
    from audioset_convnext_inf_b200.engine import fold_layernorm_into_pwconv1
    C = 384
    y, x, w1, w2, b1, b2, gamma, lw, lb = _rand_mlp(C, M, seed=M, offset=3.0)
    f = fold_layernorm_into_pwconv1(w1.cpu(), b1.cpu(), lw.cpu(), lb.cpu())
    w1f, s1, b1f = (f[k].to(DEV) for k in ("w1f", "s1", "b1f"))
    yd = y.double()
    mean = yd.mean(1, keepdim=True)
    rstd = 1.0 / torch.sqrt(yd.var(1, unbiased=False, keepdim=True) + 1e-6)
    G = yd @ w1f.double().t()
    pre = rstd * G - mean * rstd * s1.double() + b1f.double()
    d_pre = (2 * C * U24 * (yd.abs() @ w1f.double().abs().t()) + G.abs() * 8 * U24) * rstd + \
        (mean * rstd * s1.double()).abs() * 8 * U24 + pre.abs() * U24
    hid = _pw1_gp(y, w1f, b1f, s1, _row_stats(y))
    _check_gemm(f"pw1_gp M={M}", hid.double(), _gelu(pre), GELU_E + 1.13 * d_pre + _gelu(pre).abs() * 2 * U24, FRAC_GELU_LIMIT)
    xg = _to_gp(x)
    N.call("acx_gemm_bf16_pw2_gp", hid.data_ptr(), w2.data_ptr(), xg.data_ptr(), M, C, 4 * C, b2.data_ptr(), gamma.data_ptr(),
           _st())
    hd, w2d, gd = hid.double(), w2.double(), gamma.double()
    acc = hd @ w2d.t() + b2.double()
    emul = x.double() + gd * acc
    d = gd * (2 * 4 * C * U24 * (hd.abs() @ w2d.abs().t()) + acc.abs() * U24) + (x.double().abs() + (gd * acc).abs()) * U24
    _check_gemm(f"pw2_gp M={M}", _from_gp(xg, M, C).double(), emul, d, FRAC_GEMM_LIMIT)


# ======================================================================================================================
# D. Stem edges, head, front-end pieces, lengths
# ======================================================================================================================
@pytest.fixture(scope="module")
def sd():
    return weights.make_state_dict("parity", 8)


def _stem_args(sd):
    w = sd["downsample_layers.0.0.weight"].reshape(96, 16).t().contiguous().to(DEV)
    return [w] + [sd[k].to(DEV) for k in ("downsample_layers.0.0.bias", "downsample_layers.0.1.weight",
                                          "downsample_layers.0.1.bias")]


def _stem_ref(lm, sd):
    """fp64 oracle stem of (B, T, 224) log-mel -> (B, H0, 56, 96)."""
    sd64 = {k: v.double() for k, v in sd.items() if k.startswith("downsample_layers.0.")}
    return O.stem(lm.double().cpu()[:, None], sd64, F64).permute(0, 2, 3, 1).to(DEV)


def _assert_stem_bf16(tag, got, ref):
    """the bound of test_stem_tensor_core_equals_cuda_core_up_to_one_bf16_ulp, against the fp64 oracle"""
    assert torch.isfinite(got).all(), f"{tag}: unwritten outputs"
    ulp = _ulp(ref)
    diff = (got - ref).abs()
    assert (diff <= 0.5 * ulp * 1.02 + 2e-5).double().mean().item() > 0.99, tag
    assert (diff <= 1.01 * ulp + 1e-4).all(), (tag, (diff / ulp).max().item())


@pytest.mark.parametrize("T", [36, 37, 38, 39, 1000, 1001, 1002, 1003])
def test_stem_every_frame_count_mod_4(sd, T):
    """acx_stem (fp32, bf16), acx_stem_gp (read back from planar) and both _ragged twins at their full length against the
    fp64 oracle stem: the bottom padding (pad = (4, 0), stride 4) lands differently for each T mod 4."""
    B = 2
    g = torch.Generator().manual_seed(T)
    lm = (torch.randn(B, T, 224, generator=g) * 2).to(DEV)
    ref = _stem_ref(lm, sd)
    H0 = (T + 4) // 4 + 1
    assert ref.shape[1] == H0
    w, b, lw, lb = _stem_args(sd)
    p = (lm.data_ptr(), w.data_ptr(), b.data_ptr(), lw.data_ptr(), lb.data_ptr())
    full = torch.full((B,), T, device=DEV, dtype=torch.int32)
    for dtype, adt in ((torch.float32, N.ACX_F32), (torch.bfloat16, N.ACX_BF16)):
        for ragged in (False, True):
            out = torch.full((B, H0, 56, 96), float("nan"), device=DEV, dtype=dtype)
            if ragged:
                N.call("acx_stem_ragged", *p, out.data_ptr(), B, T, 224, adt, full.data_ptr(), _st())
            else:
                N.call("acx_stem", *p, out.data_ptr(), B, T, 224, adt, _st())
            if dtype == torch.float32:
                assert ((out.double() - ref).abs() <= 2e-5 + 1e-5 * ref.abs()).all(), (ragged, (out.double() - ref).abs().max().item())
            else:
                _assert_stem_bf16(f"stem bf16 ragged={ragged}", out.double(), ref)
    M = B * H0 * 56
    Mp = (M + 127) // 128 * 128
    for ragged in (False, True):
        og = torch.full((12, Mp, 8), float("nan"), device=DEV, dtype=torch.bfloat16)
        if ragged:
            N.call("acx_stem_gp_ragged", *p, og.data_ptr(), B, T, 224, full.data_ptr(), _st())
        else:
            N.call("acx_stem_gp", *p, og.data_ptr(), B, T, 224, _st())
        _assert_stem_bf16(f"stem_gp ragged={ragged}", _from_gp(og, M, 96).view(B, H0, 56, 96).double(), ref)
        assert torch.isnan(og[:, M:].float()).all(), "wrote into the plane padding past M"


def test_stem_ragged_each_clip_its_own_length(sd):
    """One ragged launch, clip b at T - b frames (every residue mod 4): the rows of each clip equal the fp64 oracle of
    the clip alone, the log-mel frames past each T_b (NaN) are never read, and nothing is written past the canvas."""
    T = 1003
    Ts = [T, T - 1, T - 2, T - 3, 37]
    B = len(Ts)
    g = torch.Generator().manual_seed(5)
    lm = (torch.randn(B, T, 224, generator=g) * 2).to(DEV)
    for b, t in enumerate(Ts):
        lm[b, t:] = float("nan")
    valid = torch.tensor(Ts, device=DEV, dtype=torch.int32)
    H0 = (T + 4) // 4 + 1
    w, b_, lw, lb = _stem_args(sd)
    p = (lm.data_ptr(), w.data_ptr(), b_.data_ptr(), lw.data_ptr(), lb.data_ptr())
    M = B * H0 * 56
    Mp = (M + 127) // 128 * 128
    og = torch.full((12, Mp, 8), float("nan"), device=DEV, dtype=torch.bfloat16)
    N.call("acx_stem_gp_ragged", *p, og.data_ptr(), B, T, 224, valid.data_ptr(), _st())
    outs = {}
    for dtype, adt in ((torch.float32, N.ACX_F32), (torch.bfloat16, N.ACX_BF16)):
        o = torch.full((M + 77, 96), float("nan"), device=DEV, dtype=dtype)
        N.call("acx_stem_ragged", *p, o.data_ptr(), B, T, 224, adt, valid.data_ptr(), _st())
        assert torch.isnan(o[M:].float()).all(), "wrote past the canvas"
        outs[dtype] = o[:M].view(B, H0, 56, 96)
    assert torch.isnan(og[:, M:].float()).all(), "wrote into the plane padding past M"
    gp = _from_gp(og, M, 96).view(B, H0, 56, 96)
    for b, t in enumerate(Ts):
        h0 = (t + 4) // 4 + 1
        ref = _stem_ref(lm[b:b + 1, :t], sd)[0]
        assert ref.shape[0] == h0
        f32 = outs[torch.float32][b, :h0].double()
        assert ((f32 - ref).abs() <= 2e-5 + 1e-5 * ref.abs()).all(), (t, (f32 - ref).abs().max().item())
        _assert_stem_bf16(f"stem_ragged bf16 T={t}", outs[torch.bfloat16][b, :h0].double(), ref)
        _assert_stem_bf16(f"stem_gp_ragged T={t}", gp[b, :h0].double(), ref)


def test_head_ragged_single_row(sd):
    """acx_head_ragged with h3 = 1, 2, 3 and the canvas height in one launch: rows past h3_b hold NaN and are never read;
    with one row the max equals the mean, so a wrong divisor of the time mean shows directly."""
    H, hs = 5, [1, 2, 3, 5, 1]
    B = len(hs)
    g = torch.Generator().manual_seed(17)
    for dtype, adt in ((torch.float32, N.ACX_F32), (torch.bfloat16, N.ACX_BF16)):
        x = torch.randn(B, H, 7, 768, generator=g).to(dtype).to(DEV)
        for b, h in enumerate(hs):
            x[b, h:] = float("nan")
        valid = torch.tensor(hs, device=DEV, dtype=torch.int32)
        t = [sd[k].to(DEV) for k in ("norm.weight", "norm.bias", "head_audioset.weight", "head_audioset.bias")]
        pooled, scene = torch.empty(B, 768, device=DEV), torch.empty(B, 768, device=DEV)
        logits, probs = torch.empty(B, 527, device=DEV), torch.empty(B, 527, device=DEV)
        N.call("acx_head_ragged", x.data_ptr(), t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(),
               pooled.data_ptr(), scene.data_ptr(), logits.data_ptr(), probs.data_ptr(), B, H, 7, 768, 527, adt,
               valid.data_ptr(), _st())
        sd64 = {k: v.double() for k, v in sd.items()}
        for b, h in enumerate(hs):
            s_ref, l_ref, p_ref = O.pool_head(x[b:b + 1, :h].double().cpu().permute(0, 3, 1, 2), sd64, F64)
            assert (scene[b].cpu().double() - s_ref[0]).abs().max() < 1e-4, (dtype, h)
            assert (logits[b].cpu().double() - l_ref[0]).abs().max() < 2e-4, (dtype, h)
            assert (probs[b].cpu().double() - p_ref[0]).abs().max() < 1e-4, (dtype, h)


def _mel_tables(sd):
    melW = sd["logmel_extractor.melW"].float().to(DEV)                      # (513, 224)
    nb, nm = melW.shape
    nz = melW != 0
    idx = torch.arange(nb, device=DEV)[:, None].expand(nb, nm)
    lo = torch.where(nz, idx, torch.full_like(idx, nb)).min(0).values
    hi = torch.where(nz, idx + 1, torch.zeros_like(idx)).max(0).values
    lo = torch.minimum(lo, hi)
    scale = (sd["bn0.weight"] / torch.sqrt(sd["bn0.running_var"] + 1e-5)).float().to(DEV)
    shift = (sd["bn0.bias"].to(DEV) - sd["bn0.running_mean"].to(DEV) * scale).float()
    return melW, lo.to(torch.int32).contiguous(), hi.to(torch.int32).contiguous(), scale.contiguous(), shift.contiguous()


def test_power_mel_log_against_fp64(sd):
    """acx_power_mel_log (the fp32-mode front end after the DFT GEMM): power -> banded mel -> 10 log10(max(., 1e-10)) ->
    bn0, against fp64 on spectra spanning 120 dB, with all-zero rows and rows below the amin clamp (exactly -100 dB)."""
    melW, lo, hi, scale, shift = _mel_tables(sd)
    nb, nm = melW.shape
    rows = 700
    g = torch.Generator().manual_seed(23)
    level = 10.0 ** (-6.0 * torch.rand(rows, 1, generator=g))                       # 0 .. -120 dB per row (amplitude)
    tilt = 10.0 ** (-3.0 * torch.rand(1, nb, generator=g))                          # and across bins
    spec = (torch.randn(rows, 2 * nb, generator=g) * level * tilt.repeat(1, 2))
    spec[::7] = 0.0                                                                 # silent frames
    spec[3::7] *= 1e-4                                                              # below amin: mel < 1e-10
    spec = spec.float().to(DEV).contiguous()
    melT = melW.t().contiguous()
    out = torch.full((rows, nm), float("nan"), device=DEV)
    N.call("acx_power_mel_log", spec.data_ptr(), 2 * nb, nb, melT.data_ptr(), lo.data_ptr(), hi.data_ptr(), scale.data_ptr(),
           shift.data_ptr(), out.data_ptr(), rows, nm, _st())
    s = spec.double()
    p = s[:, :nb] ** 2 + s[:, nb:] ** 2
    mel = p @ melW.double()
    db = 10.0 * torch.log10(mel.clamp_min(1e-10))
    ref = db * scale.double() + shift.double()
    nterm = (hi - lo).double().clamp_min(1)
    d_db = 10.0 / math.log(10.0) * (nterm + 4) * 2 * U24 + db.abs() * 4 * U24 + 1e-6    # mel sum + log10f, in dB
    bound = scale.double().abs() * d_db + (db * scale.double()).abs() * 2 * U24 + shift.double().abs() * 2 * U24
    err = (out.double() - ref).abs()
    print(f"  power_mel_log: max |err| {err.max().item():.3e}, max err / bound {(err / bound).max().item():.3f}")
    assert (err <= bound).all(), (err / bound).max().item()
    floor = -100.0 * scale.double() + shift.double()
    assert ((out.double()[::7] - floor).abs() <= bound[::7]).all()                  # amin clamp on silent frames


# lengths: T = L / 320 + 1 and h0 = (T + 4) / 4 + 1, h1 = h0 / 2, h2 = h1 / 2, h3 = h2 / 2
E2E_LENGTHS = [7360,     # MIN_RAGGED_LEN: T = 24 (0 mod 4), h = 8 4 2 1
               8961,     # T = 29 (1), h = 9 4 2 1
               13120,    # T = 42 (2), h = 12 6 3 1
               17380,    # T = 55 (3), h = 15 7 3 1
               22080,    # T = 70 (2), h = 19 9 4 2
               31680]    # T = 100 (0), h = 27 13 6 3


@pytest.fixture(scope="module")
def models(parity_sd):
    import audioset_convnext_inf_b200 as acx
    out = {}
    for prec in ("fp32", "bf16"):
        m = acx.convnext_tiny(pretrained=False, strict=False, drop_path_rate=0.0, after_stem_dim=[252, 56])
        m.load_state_dict(parity_sd, strict=True)
        out[prec] = m.to(DEV).eval().set_precision(prec)
    return out


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("L", E2E_LENGTHS)
def test_end_to_end_lengths_against_fp64_oracle(models, parity_sd, prec, L):
    """The model at clip lengths with T = 0, 2, 3 (mod 4), odd and even h1 / h2, MIN_RAGGED_LEN and 8961, against the fp64
    oracle (pinned to the reference by tests/test_oracle.py) with the golden tolerances of tests/test_gpu_model.py."""
    w = weights.make_waveforms(2, n_samples=L, kind="noise", seed=L)
    m = models[prec]
    res = m.forward_all(w.to(DEV))
    sd64 = {k: v.double() for k, v in parity_sd.items()}
    ref = O.forward(w.double(), sd64, F64)
    frame_ref = O.forward_frame_embeddings(w.double(), sd64, F64)
    scene_ref = O.forward_scene_embeddings(w.double(), sd64, F64)
    t = TOL[prec]
    fr = res["frame_embeddings"].cpu().double()
    assert fr.shape == frame_ref.shape
    d = {k: (res[k].cpu().double() - r).abs().max().item()
         for k, r in (("clipwise_logits", ref["clipwise_logits"]), ("scene_embeddings", scene_ref))}
    d["frame"] = (fr - frame_ref).abs().max().item()
    print(f"  [{prec}] L={L}: " + " ".join(f"{k} {v:.2e}" for k, v in d.items()))
    assert d["clipwise_logits"] < t["logits"] and d["scene_embeddings"] < t["scene"] and d["frame"] < t["frame"], d
