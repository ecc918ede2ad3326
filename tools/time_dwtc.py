"""Times acx_dwconv_tc / acx_layernorm_rows / acx_dwconv_ln per stage on 64 clips of 10 s (CUDA events, L2 flushed by
rotating buffers).  python tools/time_dwtc.py"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from audioset_convnext_inf_b200 import _native as N  # noqa: E402

DEV = "cuda:0"
st = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
B = 64
for stage, (C, H, W) in enumerate([(96, 252, 56), (192, 126, 28), (384, 63, 14), (768, 31, 7)]):
    xs = [torch.randn(B, H, W, C, device=DEV).to(torch.bfloat16) for _ in range(3)]
    v = torch.empty_like(xs[0])
    y = torch.empty_like(xs[0])
    w = (torch.randn(49, C, device=DEV) * 0.05).to(torch.bfloat16)
    b = torch.zeros(C, device=DEV)
    lw, lb = torch.ones(C, device=DEV), torch.zeros(C, device=DEV)

    def t(fn, iters=12):
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters * 1e3

    tc = t(lambda i: N.call("acx_dwconv_tc", xs[i % 3].data_ptr(), w.data_ptr(), b.data_ptr(), v.data_ptr(), B, H, W, C, st()))
    ln = t(lambda i: N.call("acx_layernorm_rows", xs[i % 3].data_ptr(), lw.data_ptr(), lb.data_ptr(), y.data_ptr(), B * H * W, C, st()))
    gp = float("nan")
    if stage < 2:
        gp = t(lambda i: N.call("acx_dwconv_tc_gp", xs[i % 3].data_ptr(), w.data_ptr(), b.data_ptr(), v.data_ptr(), B, H, W, C, st()))
        tr = t(lambda i: N.call("acx_gp_transpose", xs[i % 3].data_ptr(), v.data_ptr(), B * H * W, C, 1, st()))
        print(f"   group-planar: dwconv_tc_gp {gp:7.1f} us   gp_transpose {tr:7.1f} us")
    old = t(lambda i: N.call("acx_dwconv_ln", xs[i % 3].data_ptr(), w.data_ptr(), b.data_ptr(), lw.data_ptr(), lb.data_ptr(),
                             y.data_ptr(), B, H, W, C, N.ACX_BF16, st()))
    print(f"stage {stage} C={C}: dwconv_tc {tc:7.1f} us   layernorm_rows {ln:7.1f} us   (sum {tc + ln:7.1f})   dwconv_ln (CUDA cores) {old:7.1f} us")
