"""Tiny launcher for ncu: runs ONE kernel family on one ResNet-50 layer shape a few times.

    ncu --set full --clock-control none --import-source on -k regex:<kernel> -s 3 -c 1 -o gpurun_out/<name> \
        python benchmarks/ncu_target.py <what> <shape-name>

what: fwd | fwd_stats | fwd_infer | dgrad | wgrad | bn_reduce | bn_apply | bn_bwd_apply | block_grad | dwconv
shape-name: one of gpu_check.BIG_SHAPES (e.g. s4_3x3_512)
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch

import gpu_check as G
from b200ddl import ops
from b200ddl.ops import conv as C

what, shape = sys.argv[1], sys.argv[2] if len(sys.argv) > 2 else "s1_1x1_64_256"
spec = {s[0]: s for s in G.BIG_SHAPES}[shape]
name, N, H, W, cin, cout, R, stride, pad = spec
x, w, Ho, Wo = G.make_conv_case(N, H, W, cin, cout, R, stride, pad)
wk = w.to(torch.bfloat16).reshape(R * R * cout, cin).contiguous()
y = torch.empty(N, Ho, Wo, cout, device="cuda", dtype=torch.bfloat16)
dy = torch.randn_like(y)
e = ops.ext("_b200_ops")
if what in ("fwd", "fwd_stats"):
    s0 = torch.zeros(cout, device="cuda"); s1 = torch.zeros(cout, device="cuda")
    op = C.ConvForward(x, wk, y, R, R, stride, pad, *( (s0, s1) if what == "fwd_stats" else (None, None)))
elif what == "dgrad":
    op = C.ConvDgrad(dy, w, torch.empty_like(x), R, R, stride, pad)
elif what == "wgrad":
    op = C.ConvWgrad(dy, x, torch.zeros(R * R * cout, cin, device="cuda"), R, R, stride, pad)
elif what == "bn_reduce":
    s0 = torch.zeros(cout, device="cuda"); s1 = torch.zeros(cout, device="cuda")
    dz = torch.empty_like(y); g2 = torch.randn_like(y); out = torch.randn_like(y)

    class _Op:
        def run(self):
            e.bn_bwd_reduce(1, dy, g2, out, y, None, None, dz, s0, s1)
    op = _Op()
elif what == "bn_apply":
    sc = torch.ones(cout, device="cuda"); sh = torch.zeros(cout, device="cuda"); out = torch.empty_like(y); res = torch.randn_like(y)

    class _Op:
        def run(self):
            e.bn_apply(y, sc, sh, res, None, None, out, True)
    op = _Op()
elif what == "bn_bwd_apply":
    sc = torch.ones(cout, device="cuda"); sh = torch.zeros(cout, device="cuda"); out = torch.empty_like(y)
    cA = torch.ones(cout, device="cuda"); cB = torch.zeros(cout, device="cuda"); cC = torch.zeros(cout, device="cuda")

    class _Op:
        def run(self):
            e.bn_bwd_apply(dy, y, sc, sh, cA, cB, cC, out)
    op = _Op()
elif what == "block_grad":
    # conv1 dgrad of a residual block with the block-gradient epilogue (kStats = 3): cin = block channels, cout = mid
    M = N * H * W
    skip = torch.randn(N, H, W, cin, device="cuda").to(torch.bfloat16)
    y3 = torch.randn(N, H, W, cin, device="cuda").to(torch.bfloat16)
    mask = torch.randint(0, 256, (M * cin // 8,), device="cuda", dtype=torch.uint8)
    s0 = torch.zeros(cin, device="cuda"); s1 = torch.zeros(cin, device="cuda")
    dz = torch.empty(N, H, W, cin, device="cuda", dtype=torch.bfloat16)
    op = C.ConvDgrad(dy, w, dz, 1, 1, 1, 0, block_grad=(skip, mask, y3, s0, s1))
elif what == "fwd_infer":
    # inference epilogue (kStats = 4): folded BatchNorm + ReLU + residual add in the GEMM epilogue (1x1 shapes take a residual)
    sc = torch.rand(cout, device="cuda") + 0.5; sh = torch.randn(cout, device="cuda") * 0.1
    res = torch.randn_like(y) if (R == 1 and stride == 1) else None
    op = C.ConvForward(x, wk, y, R, R, stride, pad, None, None, epilogue=(sc, sh, "relu", res))
elif what == "dwconv":
    # MobileNetV2 depthwise 3x3 + folded BN + ReLU6 on the layer's INPUT shape (channels = cin)
    wd = torch.randn(9, cin, device="cuda"); sc = torch.rand(cin, device="cuda") + 0.5; sh = torch.randn(cin, device="cuda") * 0.1
    out = torch.empty(N, (H - 1) // stride + 1, (W - 1) // stride + 1, cin, device="cuda", dtype=torch.bfloat16)

    class _Op:
        def run(self):
            e.dwconv3x3(x, wd, sc, sh, out, stride)
    op = _Op()
else:
    raise SystemExit(f"unknown target {what}")
for _ in range(6):
    op.run()
torch.cuda.synchronize()
print("done", what, shape)
