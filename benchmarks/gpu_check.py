"""Kernel-by-kernel numerics + timing checks on a real B200 (run through gpurun).

    python benchmarks/gpu_check.py <case> [<case> ...]

Every case compares a hand-written sm_100a kernel against a plain PyTorch fp32 reference of the same op and
prints one ``CHECK <name> ... PASS|FAIL`` line; timing cases print ``TIME`` lines (CUDA events, warm-up, median).
The shell driver (benchmarks/run_gpu_checks.sh) runs each case in its own process under ``timeout`` so that a
hung kernel cannot take the whole GPU call down.
"""
from __future__ import annotations

import os
import sys
import time
import traceback

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch

import b200ddl  # noqa: F401
from b200ddl import ops
from b200ddl.ops import conv as C

DEV = "cuda"


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    a = a.float()
    b = b.float()
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


def report(name: str, err: float, tol: float, extra: str = "") -> bool:
    ok = err == err and err <= tol
    print(f"CHECK {name} err={err:.3e} tol={tol:.1e} {extra} {'PASS' if ok else 'FAIL'}", flush=True)
    return ok


def time_fn(fn, iters=20, warmup=5, flush=None):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        s = torch.cuda.Event(enable_timing=True)
        e = torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    ts.sort()
    return ts[len(ts) // 2]


def make_conv_case(N, H, W, cin, cout, R, stride, pad, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(N, H, W, cin, device=DEV, generator=g).to(torch.bfloat16)
    w = (torch.randn(R * R, cout, cin, device=DEV, generator=g) * (1.0 / (R * R * cin) ** 0.5))
    Ho = (H + 2 * pad - R) // stride + 1
    Wo = (W + 2 * pad - R) // stride + 1
    return x, w, Ho, Wo


CONV_SHAPES = [
    # name, N, H, W, cin, cout, R, stride, pad
    ("1x1_64_256_56", 8, 56, 56, 64, 256, 1, 1, 0),
    ("1x1_256_64_56", 8, 56, 56, 256, 64, 1, 1, 0),
    ("1x1_512_2048_7", 32, 7, 7, 512, 2048, 1, 1, 0),
    ("1x1_1024_256_14", 16, 14, 14, 1024, 256, 1, 1, 0),
    ("3x3_64_64_56", 4, 56, 56, 64, 64, 3, 1, 1),
    ("3x3_128_128_28", 8, 28, 28, 128, 128, 3, 1, 1),
    ("3x3_256_256_14", 8, 14, 14, 256, 256, 3, 1, 1),
    ("3x3_512_512_7", 16, 7, 7, 512, 512, 3, 1, 1),
    ("3x3s2_128_128_56", 4, 56, 56, 128, 128, 3, 2, 1),
    ("3x3s2_512_512_14", 8, 14, 14, 512, 512, 3, 2, 1),
    ("1x1s2_256_512_56", 4, 56, 56, 256, 512, 1, 2, 0),
]


def case_conv_fwd():
    ok = True
    for name, N, H, W, cin, cout, R, stride, pad in CONV_SHAPES:
        try:
            x, w, Ho, Wo = make_conv_case(N, H, W, cin, cout, R, stride, pad)
            wk = w.to(torch.bfloat16).reshape(R * R * cout, cin).contiguous()
            y = torch.empty(N, Ho, Wo, cout, device=DEV, dtype=torch.bfloat16)
            ssum = torch.zeros(cout, device=DEV)
            ssq = torch.zeros(cout, device=DEV)
            op = C.ConvForward(x, wk, y, R, R, stride, pad, ssum, ssq)
            op.run()
            torch.cuda.synchronize()
            ref = C.conv_reference(x, w.to(torch.bfloat16), R, R, stride, pad)
            ok &= report(f"conv_fwd/{name}", rel_err(y, ref), 1.5e-2, f"box={op.box} grid={op.plan.grid} bn={op.plan.block_n}")
            rs = ref.sum(dim=(0, 1, 2))
            rq = (ref * ref).sum(dim=(0, 1, 2))
            ok &= report(f"conv_fwd_stats_sum/{name}", float((ssum - rs).abs().max() / (rs.abs().max() + 1e-6)), 2e-2)
            ok &= report(f"conv_fwd_stats_sq/{name}", float((ssq - rq).abs().max() / (rq.abs().max() + 1e-6)), 2e-2)
        except Exception:
            ok = False
            print(f"CHECK conv_fwd/{name} EXCEPTION FAIL\n{traceback.format_exc()}", flush=True)
    return ok


def case_conv_dgrad():
    ok = True
    for name, N, H, W, cin, cout, R, stride, pad in CONV_SHAPES:
        try:
            x, w, Ho, Wo = make_conv_case(N, H, W, cin, cout, R, stride, pad)
            g = torch.Generator(device=DEV).manual_seed(1)
            dy = torch.randn(N, Ho, Wo, cout, device=DEV, generator=g).to(torch.bfloat16)
            dx = torch.full((N, H, W, cin), 7.0, device=DEV, dtype=torch.bfloat16)
            op = C.ConvDgrad(dy, w, dx, R, R, stride, pad)
            op.run()
            torch.cuda.synchronize()
            wt = C.weight_from_kernel_layout(w.to(torch.bfloat16).float(), R, R)
            ref = torch.nn.grad.conv2d_input((N, cin, H, W), wt, dy.float().permute(0, 3, 1, 2), stride=stride,
                                             padding=pad).permute(0, 2, 3, 1)
            ok &= report(f"conv_dgrad/{name}", rel_err(dx, ref), 1.5e-2, f"parts={len(op.parts)}")
            if stride == 1:
                # fused BatchNorm-backward reduction in the dgrad epilogue
                yb = torch.randn(N, H, W, cin, device=DEV, generator=g).to(torch.bfloat16)
                sc = torch.rand(cin, device=DEV, generator=g) + 0.5
                sh = torch.randn(cin, device=DEV, generator=g) * 0.5
                s_dz = torch.zeros(cin, device=DEV); s_dzy = torch.zeros(cin, device=DEV)
                dx2 = torch.empty_like(dx)
                op2 = C.ConvDgrad(dy, w, dx2, R, R, stride, pad, bwd_stats=(yb, sc, sh, s_dz, s_dzy))
                op2.run()
                torch.cuda.synchronize()
                mask = (yb.float() * sc + sh) > 0
                dzr = dx2.float() * mask
                ok &= report(f"conv_dgrad_fused_dx/{name}", rel_err(dx2, ref), 1.5e-2)
                ok &= report(f"conv_dgrad_fused_sum_dz/{name}", float((s_dz - dzr.sum((0, 1, 2))).abs().max() / (dzr.sum((0, 1, 2)).abs().max() + 1e-6)), 2e-3)
                r2 = (dzr * yb.float()).sum((0, 1, 2))
                ok &= report(f"conv_dgrad_fused_sum_dzy/{name}", float((s_dzy - r2).abs().max() / (r2.abs().max() + 1e-6)), 2e-3)
        except Exception:
            ok = False
            print(f"CHECK conv_dgrad/{name} EXCEPTION FAIL\n{traceback.format_exc()}", flush=True)
    return ok


def case_conv_wgrad():
    ok = True
    for name, N, H, W, cin, cout, R, stride, pad in CONV_SHAPES:
        try:
            x, w, Ho, Wo = make_conv_case(N, H, W, cin, cout, R, stride, pad)
            g = torch.Generator(device=DEV).manual_seed(2)
            dy = torch.randn(N, Ho, Wo, cout, device=DEV, generator=g).to(torch.bfloat16)
            dw = torch.zeros(R * R * cout, cin, device=DEV)
            op = C.ConvWgrad(dy, x, dw, R, R, stride, pad)
            op.run()
            torch.cuda.synchronize()
            ref = torch.nn.grad.conv2d_weight(x.float().permute(0, 3, 1, 2), (cout, cin, R, R),
                                              dy.float().permute(0, 3, 1, 2), stride=stride, padding=pad)
            ref = C.weight_to_kernel_layout(ref).reshape(R * R * cout, cin)
            ok &= report(f"conv_wgrad/{name}", rel_err(dw, ref), 1.0e-2,
                         f"box={op.box} units={op.plan.units} stages={op.plan.stages}")
        except Exception:
            ok = False
            print(f"CHECK conv_wgrad/{name} EXCEPTION FAIL\n{traceback.format_exc()}", flush=True)
    return ok


def case_elementwise():
    e = ops.ext("_b200_ops")
    ok = True
    g = torch.Generator(device=DEV).manual_seed(3)
    for C_ in (64, 256, 2048):
        M = 4096 + 64
        y = torch.randn(M, C_, device=DEV, generator=g).to(torch.bfloat16)
        res = torch.randn(M, C_, device=DEV, generator=g).to(torch.bfloat16)
        gamma = torch.rand(C_, device=DEV, generator=g) + 0.5
        beta = torch.randn(C_, device=DEV, generator=g)
        s = torch.zeros(C_, device=DEV); q = torch.zeros(C_, device=DEV)
        e.channel_stats(y, s, q)
        yf = y.float()
        ok &= report(f"channel_stats_sum/C{C_}", rel_err(s, yf.sum(0)), 1e-3)
        ok &= report(f"channel_stats_sq/C{C_}", rel_err(q, (yf * yf).sum(0)), 1e-3)
        rm = torch.zeros(C_, device=DEV); rv = torch.ones(C_, device=DEV)
        mean = torch.empty(C_, device=DEV); invstd = torch.empty(C_, device=DEV)
        scale = torch.empty(C_, device=DEV); shift = torch.empty(C_, device=DEV)
        e.bn_finalize(s, q, float(M), gamma, beta, rm, rv, 0.1, 1e-5, mean, invstd, scale, shift, True)
        mref = yf.mean(0); vref = yf.var(0, unbiased=False)
        ok &= report(f"bn_finalize_mean/C{C_}", float((mean - mref).abs().max()), 1e-3)
        ok &= report(f"bn_finalize_invstd/C{C_}", rel_err(invstd, (vref + 1e-5).rsqrt()), 2e-3)
        ok &= report(f"bn_finalize_zeroed/C{C_}", float(s.abs().max() + q.abs().max()), 0.0)
        out = torch.empty_like(y)
        mask = torch.zeros(M * C_ // 8, device=DEV, dtype=torch.uint8)
        e.bn_apply(y, scale, shift, res, None, None, out, True, mask)
        ref = torch.relu((yf - mref) * (vref + 1e-5).rsqrt() * gamma + beta + res.float())
        ok &= report(f"bn_apply_relu_res/C{C_}", rel_err(out, ref), 1.5e-2)
        bits = (out.float() > 0).view(M, C_ // 8, 8).to(torch.int32)
        packed = (bits * (2 ** torch.arange(8, device=DEV, dtype=torch.int32))).sum(-1).to(torch.uint8).view(-1)
        ok &= report(f"bn_apply_mask_bits/C{C_}", float((packed != mask).float().mean()), 0.0)
        s4 = torch.zeros(C_, device=DEV); s4y = torch.zeros(C_, device=DEV); dz4 = torch.empty_like(y)
        g4 = torch.randn(M, C_, device=DEV, generator=g).to(torch.bfloat16)
        e.bn_bwd_reduce(4, g4, None, mask, y, None, None, dz4, s4, s4y)
        ok &= report(f"bn_bwd_reduce_mode4/C{C_}", rel_err(dz4, g4.float() * (out.float() > 0)), 1e-2)
        # backward
        gout = torch.randn(M, C_, device=DEV, generator=g).to(torch.bfloat16)
        sdz = torch.zeros(C_, device=DEV); sdzy = torch.zeros(C_, device=DEV)
        dz = torch.empty_like(y)
        e.bn_bwd_reduce(1, gout, None, out, y, None, None, dz, sdz, sdzy)
        dz_ref = gout.float() * (out.float() > 0)
        ok &= report(f"bn_bwd_reduce_dz/C{C_}", rel_err(sdz, dz_ref.sum(0)), 2e-3)
        ok &= report(f"bn_bwd_reduce_dzy/C{C_}", rel_err(sdzy, (dz_ref * yf).sum(0)), 2e-3)
        ok &= report(f"bn_bwd_dz/C{C_}", rel_err(dz, dz_ref), 1e-2)
        dgamma = torch.empty(C_, device=DEV); dbeta = torch.empty(C_, device=DEV)
        cA = torch.empty(C_, device=DEV); cB = torch.empty(C_, device=DEV); cC = torch.empty(C_, device=DEV)
        e.bn_bwd_coeffs(sdz, sdzy, gamma, mean, invstd, float(M), dgamma, dbeta, cA, cB, cC)
        dy = torch.empty_like(y)
        e.bn_bwd_apply(dz, y, None, None, cA, cB, cC, dy)
        # mode 2: same BN+ReLU without residual, mask recomputed from y
        out2 = torch.empty_like(y)
        e.bn_apply(y, scale, shift, None, None, None, out2, True)
        s2 = torch.zeros(C_, device=DEV); s2y = torch.zeros(C_, device=DEV)
        e.bn_bwd_reduce(2, gout, None, None, y, scale, shift, None, s2, s2y)
        dz2_ref = gout.float() * (out2.float() > 0)
        ok &= report(f"bn_bwd_reduce_mode2/C{C_}", rel_err(s2, dz2_ref.sum(0)), 2e-3)
        dg2 = torch.empty(C_, device=DEV); db2 = torch.empty(C_, device=DEV)
        e.bn_bwd_coeffs(s2, s2y, gamma, mean, invstd, float(M), dg2, db2, cA, cB, cC)
        dy2 = torch.empty_like(y)
        e.bn_bwd_apply(gout, y, scale, shift, cA, cB, cC, dy2)
        yr2 = yf.clone().requires_grad_(True)
        torch.relu(torch.nn.functional.batch_norm(yr2, None, None, gamma, beta, True, 0.1, 1e-5)).backward(gout.float())
        ok &= report(f"bn_bwd_dy_mode2/C{C_}", rel_err(dy2, yr2.grad), 2e-2)
        # mode 3: no ReLU
        s3 = torch.zeros(C_, device=DEV); s3y = torch.zeros(C_, device=DEV)
        e.bn_bwd_reduce(3, gout, None, None, y, None, None, None, s3, s3y)
        e.bn_bwd_coeffs(s3, s3y, gamma, mean, invstd, float(M), dg2, db2, cA, cB, cC)
        dy3 = torch.empty_like(y)
        e.bn_bwd_apply(gout, y, None, None, cA, cB, cC, dy3)
        yr3 = yf.clone().requires_grad_(True)
        torch.nn.functional.batch_norm(yr3, None, None, gamma, beta, True, 0.1, 1e-5).backward(gout.float())
        ok &= report(f"bn_bwd_dy_mode3/C{C_}", rel_err(dy3, yr3.grad), 2e-2)
        # autograd reference
        yr = yf.clone().requires_grad_(True)
        gr = gamma.clone().requires_grad_(True); br = beta.clone().requires_grad_(True)
        o = torch.relu(torch.nn.functional.batch_norm(yr, None, None, gr, br, True, 0.1, 1e-5) + res.float())
        o.backward(gout.float())
        ok &= report(f"bn_bwd_dy/C{C_}", rel_err(dy, yr.grad), 2e-2)
        ok &= report(f"bn_bwd_dgamma/C{C_}", rel_err(dgamma, gr.grad), 1e-2)
        ok &= report(f"bn_bwd_dbeta/C{C_}", rel_err(dbeta, br.grad), 1e-2)
    # maxpool
    x = torch.relu(torch.randn(4, 16, 16, 64, device=DEV, generator=g)).to(torch.bfloat16)
    out = torch.empty(4, 8, 8, 64, device=DEV, dtype=torch.bfloat16)
    idx = torch.empty(4, 8, 8, 64, device=DEV, dtype=torch.uint8)
    e.maxpool_fwd(x, out, idx)
    xr = x.float().permute(0, 3, 1, 2).clone().requires_grad_(True)
    pr = torch.nn.functional.max_pool2d(xr, 3, 2, 1)
    ok &= report("maxpool_fwd", rel_err(out, pr.permute(0, 2, 3, 1)), 0.0)
    go = torch.randn(4, 8, 8, 64, device=DEV, generator=g).to(torch.bfloat16)
    go2 = torch.randn(4, 8, 8, 64, device=DEV, generator=g).to(torch.bfloat16)
    dx = torch.empty_like(x)
    e.maxpool_bwd(idx, go, go2, dx)
    pr.backward((go.float() + go2.float()).permute(0, 3, 1, 2))
    ok &= report("maxpool_bwd", rel_err(dx, xr.grad.permute(0, 2, 3, 1)), 1e-2)
    # fused BN + ReLU + max-pool
    yb = torch.randn(4, 16, 16, 64, device=DEV, generator=g).to(torch.bfloat16)
    scb = torch.rand(64, device=DEV, generator=g) + 0.5
    shb = torch.randn(64, device=DEV, generator=g) * 0.3
    ab = torch.empty_like(yb)
    e.bn_apply(yb, scb, shb, None, None, None, ab, True)
    p_ref = torch.empty(4, 8, 8, 64, device=DEV, dtype=torch.bfloat16); i_ref = torch.empty(4, 8, 8, 64, device=DEV, dtype=torch.uint8)
    e.maxpool_fwd(ab, p_ref, i_ref)
    p_f = torch.empty_like(p_ref); i_f = torch.empty_like(i_ref)
    e.bn_relu_maxpool_fwd(yb, scb, shb, p_f, i_f)
    ok &= report("bn_relu_maxpool_fwd", rel_err(p_f, p_ref), 0.0)
    ok &= report("bn_relu_maxpool_idx", float((i_f != i_ref).float().mean()), 0.0)
    # gap
    x = torch.randn(8, 7, 7, 2048, device=DEV, generator=g).to(torch.bfloat16)
    out = torch.empty(8, 2048, device=DEV, dtype=torch.bfloat16)
    e.gap_fwd(x, out, 0.0, 0)
    ok &= report("gap_fwd", rel_err(out, x.float().mean(dim=(1, 2))), 1e-2)
    go = torch.randn(8, 2048, device=DEV, generator=g).to(torch.bfloat16)
    dx = torch.empty_like(x)
    e.gap_bwd(go, dx, 0.0, 0)
    ok &= report("gap_bwd", rel_err(dx, (go.float() / 49)[:, None, None, :].expand(8, 7, 7, 2048)), 1e-2)
    out_d = torch.empty_like(out)
    e.gap_fwd(x, out_d, 0.5, 1234)
    keep = (out_d.float() != 0).float().mean().item()
    ok &= report("gap_dropout_keep_rate", abs(keep - 0.5), 0.05)
    # softmax ce
    for K in (5, 1000):
        B = 256
        logits = torch.randn(B, K, device=DEV, generator=g) * 3
        labels = torch.randint(0, K, (B,), device=DEV, generator=g)
        dl = torch.empty_like(logits); lr_ = torch.empty(B, device=DEV); st = torch.zeros(2, device=DEV)
        e.softmax_ce(logits, labels, dl, lr_, st, 1.0 / B)
        lg = logits.clone().requires_grad_(True)
        loss = torch.nn.functional.cross_entropy(lg, labels)
        loss.backward()
        ok &= report(f"softmax_ce_loss/K{K}", abs(st[0].item() / B - loss.item()), 1e-4)
        ok &= report(f"softmax_ce_grad/K{K}", rel_err(dl, lg.grad), 1e-3)
        acc = (logits.argmax(1) == labels).float().sum().item()
        ok &= report(f"softmax_ce_acc/K{K}", abs(st[1].item() - acc), 0.0)
    # bilinear resize (half-pixel centres, no antialias - tf.image.resize / F.interpolate(align_corners=False))
    for (H_, W_, OH, OW) in ((64, 48, 32, 32), (40, 40, 96, 96), (224, 224, 224, 224)):
        xs = torch.randint(0, 256, (3, H_, W_, 3), device=DEV, dtype=torch.uint8, generator=g)
        od = torch.empty(3, OH, OW, 3, device=DEV, dtype=torch.uint8)
        e.resize_bilinear_u8(xs, od)
        ref_r = torch.nn.functional.interpolate(xs.permute(0, 3, 1, 2).float(), size=(OH, OW), mode="bilinear",
                                                align_corners=False).permute(0, 2, 3, 1)
        ok &= report(f"resize_bilinear_u8/{H_}x{W_}->{OH}x{OW}", float((od.float() - ref_r).abs().max()), 1.0, "(max abs diff in uint8 steps)")
    # optimizers
    n = 4096 * 4
    p = torch.randn(n, device=DEV, generator=g); gr = torch.randn(n, device=DEV, generator=g)
    hyper = torch.tensor([0.1, 0.9, 0.999, 1e-8, 1e-4, 1.0, 1 - 0.9, 1 - 0.999], device=DEV)
    pr_ = p.clone().requires_grad_(True)
    opt = torch.optim.SGD([pr_], lr=0.1, momentum=0.9, weight_decay=1e-4)
    mom = torch.zeros(n, device=DEV); p16 = torch.empty(n, device=DEV, dtype=torch.bfloat16)
    pm = p.clone()
    for _ in range(3):
        pr_.grad = gr.clone(); opt.step()
        e.sgd_step(pm, gr, mom, p16, hyper, False)
    ok &= report("sgd_step", rel_err(pm, pr_.detach()), 1e-5)
    ok &= report("sgd_step_bf16", rel_err(p16, pm), 1e-2)
    pr_ = p.clone().requires_grad_(True)
    opt = torch.optim.Adam([pr_], lr=0.1, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4)
    pm = p.clone(); m = torch.zeros(n, device=DEV); v = torch.zeros(n, device=DEV)
    for t in range(1, 4):
        pr_.grad = gr.clone(); opt.step()
        hyper[6] = 1 - 0.9 ** t; hyper[7] = 1 - 0.999 ** t
        e.adam_step(pm, gr, m, v, None, hyper)
    ok &= report("adam_step", rel_err(pm, pr_.detach()), 1e-3)
    pr_ = p.clone().requires_grad_(True)
    opt = torch.optim.Adadelta([pr_], lr=1.0, rho=0.9, eps=1e-6)
    pm = p.clone(); sq = torch.zeros(n, device=DEV); ac = torch.zeros(n, device=DEV)
    h2 = torch.tensor([1.0, 0.0, 0.9, 1e-6, 0.0, 1.0, 1.0, 1.0], device=DEV)
    for t in range(3):
        pr_.grad = gr.clone(); opt.step()
        e.adadelta_step(pm, gr, sq, ac, None, h2)
    ok &= report("adadelta_step", rel_err(pm, pr_.detach()), 1e-3)
    return ok


BIG_SHAPES = [
    # ResNet-50 @ batch 256 layer shapes: name, N, H, W, cin, cout, R, stride, pad
    ("s1_1x1_64_256", 256, 56, 56, 64, 256, 1, 1, 0),
    ("s1_1x1_256_64", 256, 56, 56, 256, 64, 1, 1, 0),
    ("s1_3x3_64", 256, 56, 56, 64, 64, 3, 1, 1),
    ("s2_1x1_128_512", 256, 28, 28, 128, 512, 1, 1, 0),
    ("s2_3x3_128", 256, 28, 28, 128, 128, 3, 1, 1),
    ("s3_1x1_256_1024", 256, 14, 14, 256, 1024, 1, 1, 0),
    ("s3_1x1_1024_256", 256, 14, 14, 1024, 256, 1, 1, 0),
    ("s3_3x3_256", 256, 14, 14, 256, 256, 3, 1, 1),
    ("s4_1x1_512_2048", 256, 7, 7, 512, 2048, 1, 1, 0),
    ("s4_3x3_512", 256, 7, 7, 512, 512, 3, 1, 1),
    ("s2_3x3s2_128", 256, 56, 56, 128, 128, 3, 2, 1),
]


def case_conv_time():
    flush = torch.empty(256 * 1024 * 1024, device=DEV, dtype=torch.uint8)
    for name, N, H, W, cin, cout, R, stride, pad in BIG_SHAPES:
        try:
            x, w, Ho, Wo = make_conv_case(N, H, W, cin, cout, R, stride, pad)
            wk = w.to(torch.bfloat16).reshape(R * R * cout, cin).contiguous()
            y = torch.empty(N, Ho, Wo, cout, device=DEV, dtype=torch.bfloat16)
            ssum = torch.zeros(cout, device=DEV); ssq = torch.zeros(cout, device=DEV)
            fwd = C.ConvForward(x, wk, y, R, R, stride, pad, ssum, ssq)
            fwd_ns = C.ConvForward(x, wk, y, R, R, stride, pad)
            dy = torch.randn_like(y)
            dx = torch.empty_like(x)
            dg = C.ConvDgrad(dy, w, dx, R, R, stride, pad)
            dw = torch.zeros(R * R * cout, cin, device=DEV)
            wg = C.ConvWgrad(dy, x, dw, R, R, stride, pad)
            xc = x.permute(0, 3, 1, 2)  # channels_last NCHW view
            wt = C.weight_from_kernel_layout(w.to(torch.bfloat16), R, R).contiguous(memory_format=torch.channels_last)
            dyc = dy.permute(0, 3, 1, 2)
            flops = 2.0 * N * Ho * Wo * cout * cin * R * R
            t_f = time_fn(fwd.run, flush=flush)
            t_fn = time_fn(fwd_ns.run, flush=flush)
            t_d = time_fn(dg.run, flush=flush)
            t_w = time_fn(wg.run, flush=flush)
            t_cf = time_fn(lambda: torch.nn.functional.conv2d(xc, wt, stride=stride, padding=pad), flush=flush)
            t_cd = time_fn(lambda: torch.nn.grad.conv2d_input(xc.shape, wt, dyc, stride=stride, padding=pad), flush=flush)
            t_cw = time_fn(lambda: torch.nn.grad.conv2d_weight(xc, wt.shape, dyc, stride=stride, padding=pad), flush=flush)
            bytes_f = (x.numel() + y.numel()) * 2
            print(f"TIME {name} fwd+stats={t_f*1e3:.0f}us fwd={t_fn*1e3:.0f}us ({flops/t_fn/1e9:.0f} TF/s, "
                  f"{bytes_f/t_fn/1e6:.0f} GB/s) cudnn_fwd={t_cf*1e3:.0f}us | dgrad={t_d*1e3:.0f}us cudnn={t_cd*1e3:.0f}us | "
                  f"wgrad={t_w*1e3:.0f}us cudnn={t_cw*1e3:.0f}us", flush=True)
        except Exception:
            print(f"TIME {name} EXCEPTION\n{traceback.format_exc()}", flush=True)
    return True


def case_engine(overlap_wgrad: bool = True, quick: bool = False, fuse_block_grad=None):
    """ResNet-50 engine forward/backward vs torchvision (same weights, fp32 reference and bf16-autocast reference).

    `overlap_wgrad` selects where the weight-gradient GEMMs are issued (side stream = the engine default, or in line);
    `quick` stops after the gradient / running-statistics checks."""
    import torchvision
    from b200ddl.models.resnet_engine import ResNet50Engine, EngineTrainStep
    from b200ddl import optim

    ok = True
    N, K = 32, 10
    eng = ResNet50Engine(batch=N, num_classes=K, zero_init_residual=False, seed=1, overlap_wgrad=overlap_wgrad,
                         fuse_block_grad=fuse_block_grad)
    print(f"INFO engine overlap_wgrad={eng.overlap_wgrad} fuse_bwd_reduce={eng.fuse_bwd_reduce} "
          f"fuse_block_grad={eng.fuse_block_grad}", flush=True)
    opt = optim.SGD(learning_rate=0.1, momentum=0.9)
    step = EngineTrainStep(eng, opt, use_graph=False)
    g = torch.Generator(device=DEV).manual_seed(5)
    x = torch.randint(0, 256, (N, 224, 224, 3), device=DEV, dtype=torch.uint8, generator=g)
    y = torch.randint(0, K, (N,), device=DEV, generator=g)
    eng.set_input(x, y)
    print("STAGE engine built", flush=True)
    ref = torchvision.models.resnet50(weights=None, num_classes=K).to(DEV)
    ref.load_state_dict({k: v.to(DEV) for k, v in eng.state_dict().items()}, strict=False)
    ref.train()
    xin = (x.permute(0, 3, 1, 2).float() / 127.5 - 1.0)
    eng.forward(training=True)
    torch.cuda.synchronize()
    print("STAGE forward done", flush=True)
    eng.backward()
    torch.cuda.synchronize()
    print("STAGE backward done", flush=True)
    loss_e, acc_e = eng.loss_and_acc()
    out = ref(xin)
    loss_r = torch.nn.functional.cross_entropy(out, y)
    loss_r.backward()
    ok &= report("engine/loss_vs_fp32", abs(loss_e - loss_r.item()) / abs(loss_r.item()), 3e-2, f"engine={loss_e:.4f} ref={loss_r.item():.4f}")
    logits_err = rel_err(eng.logits, out)
    ref16 = torchvision.models.resnet50(weights=None, num_classes=K).to(DEV)
    ref16.load_state_dict({k: v.to(DEV) for k, v in eng.state_dict().items()}, strict=False)
    ref16.train()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out16 = ref16(xin)
    loss16 = torch.nn.functional.cross_entropy(out16.float(), y)
    loss16.backward()
    print(f"INFO torch-bf16-autocast loss={loss16.item():.4f} logits_err_vs_fp32={rel_err(out16, out):.3e}", flush=True)
    ok &= report("engine/logits_vs_fp32", logits_err, 1.25 * rel_err(out16, out) + 2e-2, "(tolerance = torch bf16 autocast's own error x1.25)")
    pr = dict(ref.named_parameters())
    p16 = dict(ref16.named_parameters())
    import math
    first_run = {}
    CANCELLING = {"layer1.0.bn1.bias", "bn1.weight"}
    for name in ["fc.weight", "fc.bias", "layer4.2.conv3.weight", "layer4.2.bn3.weight", "layer4.0.downsample.0.weight",
                 "layer3.0.conv2.weight", "layer2.0.conv2.weight", "layer2.1.conv1.weight", "layer1.0.conv1.weight",
                 "layer1.0.conv2.weight", "layer1.0.bn1.bias", "bn1.weight", "conv1.weight"]:
        ge = eng.g(name).detach().float()
        if name == "fc.weight":
            ge = ge[:K]  # the engine stores the class dimension zero-padded to a GEMM-friendly size
        if name.endswith("conv1.weight") or "conv" in name or "downsample.0" in name:
            k = int(round(math.sqrt(ge.shape[0])))
            ge = C.weight_from_kernel_layout(ge, k, k)
        gr = pr[name].grad.float()
        g16 = p16[name].grad.float()
        cos = torch.nn.functional.cosine_similarity(ge.flatten(), gr.flatten(), dim=0).item()
        cos16 = torch.nn.functional.cosine_similarity(g16.flatten(), gr.flatten(), dim=0).item()
        nr = (ge.norm() / (gr.norm() + 1e-12)).item()
        nr16 = (g16.norm() / (gr.norm() + 1e-12)).item()
        # distance to the fp32 gradient, ours vs torch's bf16 autocast, both relative to |g_fp32|
        d_e = ((ge - gr).norm() / (gr.norm() + 1e-12)).item()
        d_16 = ((g16 - gr).norm() / (gr.norm() + 1e-12)).item()
        first_run[name] = ge.clone()
        # The well-conditioned criterion: we must be as close to the fp32 gradient as torch's bf16 autocast is.
        # Measured over 6 runs: ratio 0.98-1.01 for conv / fc / late-BN tensors, 0.85-1.10 for the two tensors below.
        cancelling = name in CANCELLING
        ok &= report(f"engine/grad_dist/{name}", d_e, (1.5 if cancelling else 1.25) * d_16 + 3e-2,
                     f"|g-g_fp32|/|g_fp32| ours={d_e:.3f} torch_bf16={d_16:.3f} ratio={d_e / (d_16 + 1e-12):.2f}")
        if cancelling:
            # A BatchNorm affine parameter whose output reaches the next batch-statistics BatchNorm through
            # ReLU -> conv only: that BatchNorm cancels per-channel shifts / scales, so the true gradient is the small
            # residue of a huge cancellation and bf16 rounding adds incoherent energy on top.  Cosine and norm are two
            # noisy projections of the distance above and neither is stable for these tensors (identical runs: norm
            # ratio 0.76 ... 1.51, cosine gap 0.80 ... 0.99; torch bf16: 1.04 / 1.13 and 0.72 / 1.10) - printed, not gated.
            print(f"INFO engine/grad_cos/{name} gap ours={1-cos:.3f} torch_bf16={1-cos16:.3f}; grad_norm ours={nr:.3f} "
                  f"torch_bf16={nr16:.3f} (cancellation residue, informational)", flush=True)
        else:
            # bf16 networks at random init are chaotic w.r.t. rounding: judge against what torch's own bf16 autocast achieves
            ok &= report(f"engine/grad_cos/{name}", 1.0 - cos, 1.25 * (1 - cos16) + 3e-2,
                         f"norm_ratio={nr:.3f} torch_bf16_cos_gap={1-cos16:.2e}")
            ok &= report(f"engine/grad_norm/{name}", abs(nr - 1.0), 0.10, f"torch_bf16={nr16:.3f}")
    # running stats
    rm = dict(ref.named_buffers())
    ok &= report("engine/running_mean/bn1", rel_err(eng.running_mean["bn1"], rm["bn1.running_mean"]), 3e-2)
    ok &= report("engine/running_var/layer3.0.bn2", rel_err(eng.running_var["layer3.0.bn2"], rm["layer3.0.bn2.running_var"]), 5e-2)
    if quick:
        return ok
    # run-to-run spread of the engine itself (fp32 atomics in the statistics / wgrad reductions are unordered): the same
    # input through forward+backward again, compared with the first run.  Diagnostic only.
    eng.forward(training=True)
    eng.backward()
    torch.cuda.synchronize()
    for name, g1 in first_run.items():
        g2 = eng.g(name).detach().float()
        if name == "fc.weight":
            g2 = g2[:K]
        if g2.shape != g1.shape:
            k = int(round(math.sqrt(g2.shape[0])))
            g2 = C.weight_from_kernel_layout(g2, k, k)
        print(f"INFO engine/self_variation/{name} rel_diff={((g2 - g1).norm() / (g1.norm() + 1e-12)).item():.3e} "
              f"norm_ratio_run2/run1={(g2.norm() / (g1.norm() + 1e-12)).item():.4f}", flush=True)
    # Is that spread ours or the network's?  The same experiment on torch alone: bf16 autocast again with every
    # BatchNorm weight (kept in fp32 by autocast, applied before the bf16 rounding - where our unordered fp32 statistics
    # sums enter) perturbed by a few fp32 ulps, compared with the first bf16 run.  (A first version perturbed the conv
    # weights by 1e-7: below one ulp and then rounded to bf16, i.e. no perturbation at all - hence the validity check.)
    ref16b = torchvision.models.resnet50(weights=None, num_classes=K).to(DEV)
    ref16b.load_state_dict(ref16.state_dict())
    ref16b.train()
    with torch.no_grad():
        gp = torch.Generator(device=DEV).manual_seed(11)
        n_changed = 0
        for m in ref16b.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                before = m.weight.clone()
                m.weight.mul_(1.0 + 3e-7 * torch.randn(m.weight.shape, device=DEV, generator=gp))
                n_changed += int((m.weight != before).sum().item())
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out16b = ref16b(xin)
    torch.nn.functional.cross_entropy(out16b.float(), y).backward()
    fwd_diff = rel_err(out16b, out16)
    print(f"INFO torch_bf16_sensitivity: {n_changed} BatchNorm weights changed by ~3e-7 relative; logits rel_diff={fwd_diff:.3e} "
          f"({'VALID' if fwd_diff > 0 else 'INVALID - the perturbation did not reach the bf16 computation'})", flush=True)
    p16b = dict(ref16b.named_parameters())
    for name in first_run:
        ga, gb = p16[name].grad.float(), p16b[name].grad.float()
        print(f"INFO torch_bf16_sensitivity_bn3e-7/{name} rel_diff={((gb - ga).norm() / (ga.norm() + 1e-12)).item():.3e}", flush=True)
    # a few optimisation steps must reduce the loss on a fixed batch (graph path)
    print("STAGE graph steps", flush=True)
    eng2 = ResNet50Engine(batch=N, num_classes=K, seed=2, overlap_wgrad=overlap_wgrad)
    step2 = EngineTrainStep(eng2, optim.SGD(learning_rate=0.05, momentum=0.9), use_graph=True)
    losses = []
    for i in range(12):
        step2.load(x, y)
        step2.run()
        losses.append(step2.result()[0])
    print("INFO graph-step losses", " ".join(f"{l:.3f}" for l in losses), flush=True)
    ok &= report("engine/loss_decreases", float(losses[-1] >= losses[0]), 0.0, f"{losses[0]:.3f}->{losses[-1]:.3f}")
    ok &= report("engine/loss_finite", float(not all(l == l and abs(l) < 1e4 for l in losses)), 0.0)
    # eval-mode forward runs and is finite
    from b200ddl.models.resnet_engine import EngineEvalStep
    ev = EngineEvalStep(eng2)
    ev.run()
    le, ae = ev.result()
    ok &= report("engine/eval_finite", float(not (le == le and le < 1e4)), 0.0, f"eval loss={le:.3f} acc={ae:.3f}")
    return ok


def case_stem():
    """7x7/2 stem conv on uint8 input: forward (+BN stats) and weight gradient vs torch."""
    ok = True
    g = torch.Generator(device=DEV).manual_seed(11)
    for N, S in ((4, 64), (16, 224), (3, 96)):
        x = torch.randint(0, 256, (N, S, S, 3), device=DEV, dtype=torch.uint8, generator=g)
        w = torch.randn(49, 64, 3, device=DEV, generator=g) * 0.08
        w16 = torch.zeros(64, 192, device=DEV, dtype=torch.bfloat16)
        C.pack_stem_weight(w, w16)
        Ho = S // 2
        y = torch.empty(N, Ho, Ho, 64, device=DEV, dtype=torch.bfloat16)
        ssum = torch.zeros(64, device=DEV); ssq = torch.zeros(64, device=DEV)
        C.StemForward(x, w16, y, ssum, ssq).run()
        torch.cuda.synchronize()
        xin = (x.float() / 127.5 - 1.0).to(torch.bfloat16).float().permute(0, 3, 1, 2)
        wt = w.to(torch.bfloat16).float().view(7, 7, 64, 3).permute(2, 3, 0, 1)
        ref = torch.nn.functional.conv2d(xin, wt, stride=2, padding=3).permute(0, 2, 3, 1)
        ok &= report(f"stem_fwd/N{N}_S{S}", rel_err(y, ref), 1.5e-2)
        ok &= report(f"stem_fwd_stats_sum/N{N}_S{S}", float((ssum - ref.sum((0, 1, 2))).abs().max() / (ref.sum((0, 1, 2)).abs().max() + 1e-6)), 2e-2)
        ok &= report(f"stem_fwd_stats_sq/N{N}_S{S}", rel_err(ssq, (ref * ref).sum((0, 1, 2))), 2e-2)
        dy = torch.randn(N, Ho, Ho, 64, device=DEV, generator=g).to(torch.bfloat16)
        dw = torch.zeros(49 * 64 * 3, device=DEV)
        C.StemWgrad(x, dy, dw).run()
        torch.cuda.synchronize()
        gref = torch.nn.grad.conv2d_weight(xin, (64, 3, 7, 7), dy.float().permute(0, 3, 1, 2), stride=2, padding=3)
        gref = gref.permute(2, 3, 0, 1).reshape(49, 64, 3)
        ok &= report(f"stem_wgrad/N{N}_S{S}", rel_err(dw.view(49, 64, 3), gref), 1e-2)
    # timing at the benchmark shape
    N, S = 256, 224
    x = torch.randint(0, 256, (N, S, S, 3), device=DEV, dtype=torch.uint8, generator=g)
    w16 = torch.zeros(64, 192, device=DEV, dtype=torch.bfloat16)
    y = torch.empty(N, 112, 112, 64, device=DEV, dtype=torch.bfloat16)
    ssum = torch.zeros(64, device=DEV); ssq = torch.zeros(64, device=DEV)
    f = C.StemForward(x, w16, y, ssum, ssq)
    dw = torch.zeros(49 * 64 * 3, device=DEV)
    wg = C.StemWgrad(x, y, dw)
    flush = torch.empty(256 * 1024 * 1024, device=DEV, dtype=torch.uint8)
    print(f"TIME stem fwd+stats={time_fn(f.run, flush=flush)*1e3:.0f}us wgrad={time_fn(wg.run, flush=flush)*1e3:.0f}us "
          f"(cuDNN path in the first profile: fwd 1465us + pad 228us, wgrad 759us)", flush=True)
    return ok



def _pack_mask(mask_bool: torch.Tensor) -> torch.Tensor:
    """[M, C] bool -> uint8 [M * C / 8], bit k of byte cv = channel cv*8 + k (the layout bn_apply writes)."""
    M, C_ = mask_bool.shape
    bits = mask_bool.view(M, C_ // 8, 8).to(torch.int32)
    return (bits * (2 ** torch.arange(8, device=mask_bool.device, dtype=torch.int32))).sum(-1).to(torch.uint8).view(-1).contiguous()


BLOCK_GRAD_SHAPES = [
    # name, N, H, block_cin (dgrad output channels), mid (dgrad K), compact skip
    ("s1_256_64", 8, 56, 256, 64, False),
    ("s2_512_128", 8, 28, 512, 128, False),
    ("s2_first_512_256_compact", 8, 28, 512, 128, True),
    ("s4_2048_512_partial_tile", 8, 7, 2048, 512, False),   # M = 392: last tile has 8 real rows
    ("s3_compact_14", 6, 14, 1024, 256, True),
    ("bench_s1_256_64_b256", 256, 56, 256, 64, False),      # the benchmark shape (M = 802,816)
    ("bench_s2_first_b256_compact", 256, 28, 512, 128, True),
]


def case_block_grad():
    """conv1-dgrad with the block-gradient epilogue (kStats = 3): dz = (dgrad + skip) * relu_mask, sum(dz), sum(dz*y3)."""
    ok = True
    e = ops.ext("_b200_ops")
    for name, N, H, cb, mid, compact in BLOCK_GRAD_SHAPES:
        try:
            g = torch.Generator(device=DEV).manual_seed(17)
            dy = torch.randn(N, H, H, mid, device=DEV, generator=g).to(torch.bfloat16)
            w = torch.randn(1, mid, cb, device=DEV, generator=g) * (1.0 / mid ** 0.5)   # conv1: cb -> mid
            hs = H // 2 if compact else H
            skip = torch.randn(N, hs, hs, cb, device=DEV, generator=g).to(torch.bfloat16)
            y3 = torch.randn(N, H, H, cb, device=DEV, generator=g).to(torch.bfloat16)
            mbool = torch.rand(N * H * H, cb, device=DEV, generator=g) > 0.45
            mask = _pack_mask(mbool)
            s_dz = torch.zeros(cb, device=DEV); s_dzy = torch.zeros(cb, device=DEV)
            dz = torch.full((N, H, H, cb), 3.0, device=DEV, dtype=torch.bfloat16)
            op = C.ConvDgrad(dy, w, dz, 1, 1, 1, 0, block_grad=(skip, mask, y3, s_dz, s_dzy))
            op.run()
            torch.cuda.synchronize()
            # reference in fp32 (bf16-rounded weights, like the kernel's operand)
            ref_g = dy.float().view(-1, mid) @ w[0].to(torch.bfloat16).float()          # [M, cb]
            if compact:
                full = torch.zeros(N, H, H, cb, device=DEV)
                full[:, 0::2, 0::2, :] = skip.float()
            else:
                full = skip.float()
            ref_dz = (ref_g + full.view(-1, cb)) * mbool
            ok &= report(f"block_grad_dz/{name}", rel_err(dz.view(-1, cb), ref_dz), 1.5e-2,
                         f"grid={op.parts[0][0].grid} stats_mode={op.parts[0][0].stats_mode}")
            dzq = dz.float().view(-1, cb)   # the sums are taken over the bf16 values that were stored
            r0 = dzq.sum(0); r1 = (dzq * y3.float().view(-1, cb)).sum(0)
            ok &= report(f"block_grad_sum_dz/{name}", float((s_dz - r0).abs().max() / (r0.abs().max() + 1e-6)), 2e-3)
            ok &= report(f"block_grad_sum_dzy/{name}", float((s_dzy - r1).abs().max() / (r1.abs().max() + 1e-6)), 2e-3)
            if N >= 256:
                flush = torch.empty(256 * 1024 * 1024, device=DEV, dtype=torch.uint8)
                # what it replaces: plain dgrad + reduce pass (mode 4) that also stores dz
                g1 = torch.empty(N, H, H, cb, device=DEV, dtype=torch.bfloat16)
                plain = C.ConvDgrad(dy, w, g1, 1, 1, 1, 0)
                dz2 = torch.empty_like(g1)
                skipd = full.to(torch.bfloat16).view(N, H, H, cb).contiguous()
                def old():
                    plain.run()
                    e.bn_bwd_reduce(4, g1, skipd, mask, y3, None, None, dz2, s_dz, s_dzy)
                t_new = time_fn(op.run, flush=flush)
                t_plain = time_fn(plain.run, flush=flush)
                t_old = time_fn(old, flush=flush)
                nbytes = (dy.numel() + skip.numel() + y3.numel() + dz.numel()) * 2 + mask.numel()
                print(f"TIME block_grad/{name} fused={t_new*1e3:.0f}us ({nbytes/t_new/1e6:.0f} GB/s algorithmic) "
                      f"plain_dgrad={t_plain*1e3:.0f}us dgrad+reduce(mode4)={t_old*1e3:.0f}us", flush=True)
        except Exception:
            ok = False
            print(f"CHECK block_grad/{name} EXCEPTION FAIL\n{traceback.format_exc()}", flush=True)
    return ok


def case_head():
    """Classifier head: FC forward / dgrad / wgrad on the tcgen05 GEMMs + softmax_ce_head + fc_bias_grad vs torch fp32."""
    ok = True
    e = ops.ext("_b200_ops")
    for N, K in ((256, 1000), (8, 5), (32, 10), (64, 200)):
        try:
            g = torch.Generator(device=DEV).manual_seed(23)
            ncp = 64 if K <= 64 else (K + 127) // 128 * 128
            pooled = torch.randn(N, 2048, device=DEV, generator=g).to(torch.bfloat16)
            wm = torch.zeros(ncp, 2048, device=DEV)
            wm[:K] = (torch.rand(K, 2048, device=DEV, generator=g) * 2 - 1) / 2048 ** 0.5 * 4
            bias = torch.randn(K, device=DEV, generator=g) * 0.1
            labels = torch.randint(0, K, (N,), device=DEV, generator=g)
            w16 = wm.to(torch.bfloat16)
            logits16 = torch.zeros(N, ncp, device=DEV, dtype=torch.bfloat16)
            C.ConvForward(pooled.view(N, 1, 1, 2048), w16, logits16.view(N, 1, 1, ncp), 1, 1, 1, 0).run()
            logits32 = torch.zeros(N, K, device=DEV); dl16 = torch.full((N, ncp), 9.0, device=DEV, dtype=torch.bfloat16)
            rows = torch.zeros(N, device=DEV); st = torch.zeros(2, device=DEV)
            e.softmax_ce_head(logits16, bias, labels, logits32, dl16, rows, st, 1.0 / N)
            torch.cuda.synchronize()
            ref_logits = pooled.float() @ w16[:K].float().t() + bias
            ok &= report(f"head_logits/N{N}_K{K}", rel_err(logits32, ref_logits), 1.5e-2)
            lg = logits32.clone().requires_grad_(True)   # CE itself is checked on the kernel's own logits
            loss = torch.nn.functional.cross_entropy(lg, labels)
            loss.backward()
            ok &= report(f"head_loss/N{N}_K{K}", abs(st[0].item() / N - loss.item()), 1e-4)
            ok &= report(f"head_acc/N{N}_K{K}", abs(st[1].item() - (logits32.argmax(1) == labels).float().sum().item()), 0.0)
            ok &= report(f"head_dlogits/N{N}_K{K}", rel_err(dl16[:, :K], lg.grad), 1e-2)
            ok &= report(f"head_dlogits_pad_zero/N{N}_K{K}", float(dl16[:, K:].float().abs().max()) if ncp > K else 0.0, 0.0)
            db = torch.zeros(K, device=DEV)
            e.fc_bias_grad(dl16, db)
            ok &= report(f"head_dbias/N{N}_K{K}", rel_err(db, dl16[:, :K].float().sum(0)), 1e-5)
            # weight gradient and data gradient on the GEMM kernels
            dw = torch.zeros(ncp, 2048, device=DEV)
            C.ConvWgrad(dl16.view(N, 1, 1, ncp), pooled.view(N, 1, 1, 2048), dw, 1, 1, 1, 0).run()
            ok &= report(f"head_wgrad/N{N}_K{K}", rel_err(dw, dl16.float().t() @ pooled.float()), 1e-2)
            dpooled = torch.zeros(N, 2048, device=DEV, dtype=torch.bfloat16)
            C.ConvDgrad(dl16.view(N, 1, 1, ncp), wm.view(1, ncp, 2048), dpooled.view(N, 1, 1, 2048), 1, 1, 1, 0).run()
            torch.cuda.synchronize()
            ok &= report(f"head_dgrad/N{N}_K{K}", rel_err(dpooled, dl16.float() @ w16.float()), 1.5e-2)
        except Exception:
            ok = False
            print(f"CHECK head/N{N}_K{K} EXCEPTION FAIL\n{traceback.format_exc()}", flush=True)
    # stem filter pack kernel vs the python permutation
    w = torch.randn(49, 64, 3, device=DEV)
    a = torch.zeros(64, 192, device=DEV, dtype=torch.bfloat16); b = torch.full((64, 192), 5.0, device=DEV, dtype=torch.bfloat16)
    C.pack_stem_weight(w, a)
    e.pack_stem_weight(w, b)
    ok &= report("pack_stem_weight", float((a.float() - b.float()).abs().max()), 0.0)
    return ok


def case_big_numerics():
    """Numerics at the BENCHMARKED shapes (batch 256: full grids, halo / resident-filter paths, 802,816-pixel M) vs fp32."""
    ok = True
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    for name, N, H, W, cin, cout, R, stride, pad in BIG_SHAPES:
        try:
            x, w, Ho, Wo = make_conv_case(N, H, W, cin, cout, R, stride, pad)
            w16 = w.to(torch.bfloat16)
            wk = w16.reshape(R * R * cout, cin).contiguous()
            y = torch.empty(N, Ho, Wo, cout, device=DEV, dtype=torch.bfloat16)
            ssum = torch.zeros(cout, device=DEV); ssq = torch.zeros(cout, device=DEV)
            op = C.ConvForward(x, wk, y, R, R, stride, pad, ssum, ssq)
            op.run()
            torch.cuda.synchronize()
            ref = C.conv_reference(x, w16, R, R, stride, pad)
            ok &= report(f"big_fwd/{name}", rel_err(y, ref), 1.5e-2, f"box={op.box} halo={op.plan.halo} res={op.plan.resident_filter}")
            yq = y.float()
            ok &= report(f"big_fwd_stats_sum/{name}", float((ssum - yq.sum((0, 1, 2))).abs().max() / (yq.sum((0, 1, 2)).abs().max() + 1e-6)), 2e-3)
            ok &= report(f"big_fwd_stats_sq/{name}", rel_err(ssq, (yq * yq).sum((0, 1, 2))), 2e-3)
            del yq
            g = torch.Generator(device=DEV).manual_seed(1)
            dy = torch.randn(N, Ho, Wo, cout, device=DEV, generator=g).to(torch.bfloat16)
            dx = torch.full((N, H, W, cin), 7.0, device=DEV, dtype=torch.bfloat16)
            C.ConvDgrad(dy, w, dx, R, R, stride, pad).run()
            torch.cuda.synchronize()
            wt = C.weight_from_kernel_layout(w16.float(), R, R)
            refd = torch.nn.grad.conv2d_input((N, cin, H, W), wt, dy.float().permute(0, 3, 1, 2), stride=stride,
                                              padding=pad).permute(0, 2, 3, 1)
            ok &= report(f"big_dgrad/{name}", rel_err(dx, refd), 1.5e-2)
            del refd
            dw = torch.zeros(R * R * cout, cin, device=DEV)
            C.ConvWgrad(dy, x, dw, R, R, stride, pad).run()
            torch.cuda.synchronize()
            refw = torch.nn.grad.conv2d_weight(x.float().permute(0, 3, 1, 2), (cout, cin, R, R),
                                               dy.float().permute(0, 3, 1, 2), stride=stride, padding=pad)
            refw = C.weight_to_kernel_layout(refw).reshape(R * R * cout, cin)
            ok &= report(f"big_wgrad/{name}", rel_err(dw, refw), 1.0e-2)
            del ref, refw, x, y, dy, dx
            torch.cuda.empty_cache()
        except Exception:
            ok = False
            print(f"CHECK big/{name} EXCEPTION FAIL\n{traceback.format_exc()}", flush=True)
    return ok



def case_fused_infer():
    """Inference epilogue (conv_igemm kStats = 4): y = act(conv * scale + shift [+ residual]) vs fp32, on flat / box / halo /
    strided plans; then the inference-built ResNet-50 engine (no BatchNorm passes) vs the training-built engine's eval path."""
    ok = True
    g = torch.Generator(device=DEV).manual_seed(41)
    for name, N, H, W, cin, cout, R, stride, pad in CONV_SHAPES + [("bench_s1_1x1_64_256_b256", 256, 56, 56, 64, 256, 1, 1, 0)]:
        try:
            x, w, Ho, Wo = make_conv_case(N, H, W, cin, cout, R, stride, pad)
            w16 = w.to(torch.bfloat16)
            wk = w16.reshape(R * R * cout, cin).contiguous()
            scale = torch.rand(cout, device=DEV, generator=g) + 0.5
            shift = torch.randn(cout, device=DEV, generator=g) * 0.5
            ref = C.conv_reference(x, w16, R, R, stride, pad) * scale + shift
            flat = (R == 1 and stride == 1)
            for act in ("relu", "relu6", "none"):
                res = torch.randn(N, Ho, Wo, cout, device=DEV, generator=g).to(torch.bfloat16) if (flat and act != "relu6") else None
                y = torch.full((N, Ho, Wo, cout), 9.0, device=DEV, dtype=torch.bfloat16)
                op = C.ConvForward(x, wk, y, R, R, stride, pad, epilogue=(scale, shift, act, res))
                op.run()
                torch.cuda.synchronize()
                r = ref + (res.float() if res is not None else 0.0)
                r = torch.relu(r) if act == "relu" else (r.clamp(0, 6) if act == "relu6" else r)
                ok &= report(f"fused_infer_conv/{name}/{act}{'+res' if res is not None else ''}", rel_err(y, r), 1.5e-2,
                             f"box={op.box} bn={op.plan.block_n} halo={op.plan.halo}")
        except Exception:
            ok = False
            print(f"CHECK fused_infer_conv/{name} EXCEPTION FAIL\n{traceback.format_exc()}", flush=True)
    # engine level: same weights / running statistics, inference build (fused epilogues) vs training build (eval mode)
    from b200ddl.models.resnet_engine import EngineEvalStep, ResNet50Engine
    N, K = 32, 10
    ref_eng = ResNet50Engine(batch=N, num_classes=K, zero_init_residual=False, seed=3)
    ref_eng.bind_grad_buffer()
    ref_eng.build(training=True)
    for n_ in ref_eng.bn_names:   # non-trivial running statistics
        ref_eng.running_mean[n_].copy_(torch.randn(ref_eng.bn_channels[n_], device=DEV, generator=g) * 0.1)
        ref_eng.running_var[n_].copy_(torch.rand(ref_eng.bn_channels[n_], device=DEV, generator=g) + 0.5)
    sd = ref_eng.state_dict()
    inf = ResNet50Engine(batch=N, num_classes=K, zero_init_residual=False, seed=99)
    inf.load_state_dict(sd)
    inf.build(training=False)
    xs = torch.randint(0, 256, (N, 224, 224, 3), device=DEV, dtype=torch.uint8, generator=g)
    ys = torch.randint(0, K, (N,), device=DEV, generator=g)
    ref_eng.set_input(xs, ys); inf.set_input(xs, ys)
    ref_eng.forward(training=False)
    ev = EngineEvalStep(inf)
    ev.run(); ev.run()
    torch.cuda.synchronize()
    print(f"INFO fused inference engine: infer_fused={inf._infer_fused} launches={len(inf._fwd)} conv plans", flush=True)
    ok &= report("fused_infer_engine/logits", rel_err(inf.logits, ref_eng.logits), 3e-2)
    ok &= report("fused_infer_engine/argmax_agree", 1.0 - float((inf.logits.argmax(1) == ref_eng.logits.argmax(1)).float().mean()), 0.1)
    # throughput of the two eval paths at the serving batch
    for label, build_training in (("bn_passes", True), ("fused_epilogues", False)):
        e2 = ResNet50Engine(batch=256, num_classes=1000, seed=5)
        if build_training:
            e2.bind_grad_buffer()
        e2.build(training=build_training)
        st = EngineEvalStep(e2)
        t = time_fn(st.run, iters=10, warmup=3)
        print(f"TIME eval_forward/{label} batch 256: {t*1e3:.0f} us = {256 / t * 1e3:.0f} images/s", flush=True)
        del e2, st
        torch.cuda.empty_cache()
    return ok



def case_mobilenet():
    """The reference's own model on native kernels: depthwise / stem kernels vs torch, then the whole frozen-base
    MobileNetV2 engine (tcgen05 pointwise convs with folded-BN epilogues) vs the torch.nn module with the same weights."""
    ok = True
    e = ops.ext("_b200_ops")
    g = torch.Generator(device=DEV).manual_seed(51)
    # depthwise 3x3 + affine + relu6
    for (N, H, C_, stride) in ((2, 14, 64, 1), (3, 28, 192, 2), (2, 7, 960, 1), (2, 7, 64, 2), (1, 13, 32, 1), (2, 112, 96, 2),
                               (1, 9, 16, 2)):
        x = torch.randn(N, H, H, C_, device=DEV, generator=g).to(torch.bfloat16)
        w = torch.randn(9, C_, device=DEV, generator=g) * 0.3
        sc = torch.rand(C_, device=DEV, generator=g) + 0.5
        sh = torch.randn(C_, device=DEV, generator=g) * 0.5
        Ho = (H - 1) // stride + 1
        out = torch.empty(N, Ho, Ho, C_, device=DEV, dtype=torch.bfloat16)
        e.dwconv3x3(x, w, sc, sh, out, stride)          # register-tiled kernel (default, 4 output pixels per thread)
        out1 = torch.empty_like(out)
        e.dwconv3x3(x, w, sc, sh, out1, stride, 1)      # one-pixel kernel
        wt = w.t().reshape(C_, 1, 3, 3)
        ref = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), wt, stride=stride, padding=1, groups=C_)
        ref = (ref * sc.view(1, -1, 1, 1) + sh.view(1, -1, 1, 1)).clamp(0, 6).permute(0, 2, 3, 1)
        ok &= report(f"dwconv3x3/N{N}_H{H}_C{C_}_s{stride}", rel_err(out, ref), 1e-2)
        ok &= report(f"dwconv3x3 tiled == one-pixel/N{N}_H{H}_C{C_}_s{stride}", 0.0 if torch.equal(out, out1) else 1.0, 0.5)
    # MobileNetV2's depthwise layers at batch 64: tiled vs one-pixel kernel
    tot = [0.0, 0.0]
    l2 = torch.empty(256 << 20, device=DEV, dtype=torch.uint8)   # written between timed launches: inputs never come from L2

    def time_op(fn):
        return time_fn(fn, iters=10, warmup=3, flush=l2) * 1e3

    for (H, C_, stride) in ((112, 32, 1), (112, 96, 2), (56, 144, 1), (56, 144, 2), (28, 192, 1), (28, 192, 2), (14, 384, 1),
                            (14, 576, 1), (14, 576, 2), (7, 960, 1)):
        Cp = (C_ + 63) // 64 * 64
        x = torch.randn(64, H, H, Cp, device=DEV, generator=g).to(torch.bfloat16)
        w = torch.randn(9, Cp, device=DEV, generator=g) * 0.3
        sc = torch.rand(Cp, device=DEV, generator=g) + 0.5
        sh = torch.randn(Cp, device=DEV, generator=g) * 0.5
        Ho = (H - 1) // stride + 1
        out = torch.empty(64, Ho, Ho, Cp, device=DEV, dtype=torch.bfloat16)
        t4 = time_op(lambda: e.dwconv3x3(x, w, sc, sh, out, stride, 4))
        t1 = time_op(lambda: e.dwconv3x3(x, w, sc, sh, out, stride, 1))
        gb = (x.numel() + out.numel()) * 2 / 1e9
        tot[0] += t4
        tot[1] += t1
        print(f"TIME dwconv3x3 b64 {H}x{H}x{Cp} s{stride}: tiled {t4:.1f} us ({gb / t4 * 1e6:.0f} GB/s)  one-pixel {t1:.1f} us", flush=True)
    print(f"TIME dwconv3x3 sum over the 10 shapes: tiled {tot[0]:.0f} us, one-pixel {tot[1]:.0f} us", flush=True)
    # stem 3x3/2 from uint8
    xs = torch.randint(0, 256, (3, 64, 64, 3), device=DEV, dtype=torch.uint8, generator=g)
    wst = torch.randn(32, 3, 3, 3, device=DEV, generator=g) * 0.2
    sc = torch.rand(32, device=DEV, generator=g) + 0.5
    sh = torch.randn(32, device=DEV, generator=g) * 0.5
    out = torch.zeros(3, 32, 32, 64, device=DEV, dtype=torch.bfloat16)
    e.mbv2_stem(xs, wst.permute(2, 3, 1, 0).reshape(27, 32).contiguous(), sc, sh, out, 1.0 / 127.5, -1.0)
    xin = (xs.float() / 127.5 - 1.0).to(torch.bfloat16).float().permute(0, 3, 1, 2)
    ref = torch.nn.functional.conv2d(xin, wst, stride=2, padding=1)
    ref = (ref * sc.view(1, -1, 1, 1) + sh.view(1, -1, 1, 1)).clamp(0, 6).permute(0, 2, 3, 1)
    ok &= report("mbv2_stem", rel_err(out[..., :32], ref), 1e-2)
    ok &= report("mbv2_stem_padding_untouched", float(out[..., 32:].float().abs().max()), 0.0)
    # whole model vs the torch module (fp32) with identical weights
    from b200ddl.models import build_model
    from b200ddl.models.mobilenet_engine import MobileNetV2Engine
    N, K = 16, 5
    eng = build_model(224, 224, 3, K, dropout=0.0, arch="mobilenetv2", batch_size=N, seed=3)
    assert isinstance(eng, MobileNetV2Engine), type(eng)
    ref = build_model(224, 224, 3, K, dropout=0.0, arch="mobilenetv2_torch", seed=3).to(DEV)
    # non-trivial BatchNorm statistics / affine so the folded epilogues are really exercised
    with torch.no_grad():
        for m in ref.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.num_features, device=DEV, generator=g) * 0.1)
                m.running_var.copy_(torch.rand(m.num_features, device=DEV, generator=g) * 0.5 + 0.75)
                m.weight.copy_(torch.rand(m.num_features, device=DEV, generator=g) * 0.5 + 0.75)
                m.bias.copy_(torch.randn(m.num_features, device=DEV, generator=g) * 0.1)
    eng.load_state_dict(ref.state_dict())
    eng.bind_grad_buffer()
    eng.build(training=True)
    x = torch.randint(0, 256, (N, 224, 224, 3), device=DEV, dtype=torch.uint8, generator=g)
    y = torch.randint(0, K, (N,), device=DEV, generator=g)
    eng.set_input(x, y)
    eng.forward(training=True)
    eng.backward()
    torch.cuda.synchronize()
    ref.train()
    logits = ref((x.permute(0, 3, 1, 2).float() / 127.5 - 1.0))
    loss = torch.nn.functional.cross_entropy(logits, y)
    loss.backward()
    feat_ref = ref.base((x.permute(0, 3, 1, 2).float() / 127.5 - 1.0)).mean(dim=(2, 3))
    ok &= report("mobilenet_engine/features", rel_err(eng.pooled, feat_ref), 6e-2, f"launches per forward ~{len(eng._plan) + 4}")
    ok &= report("mobilenet_engine/logits", rel_err(eng.logits, logits), 6e-2)
    le, _ = eng.loss_and_acc()
    ok &= report("mobilenet_engine/loss", abs(le - loss.item()) / abs(loss.item()), 3e-2, f"engine={le:.4f} torch={loss.item():.4f}")
    gw = eng.g("fc.weight")[:K]
    cos = torch.nn.functional.cosine_similarity(gw.flatten(), ref.fc.weight.grad.flatten(), dim=0).item()
    ok &= report("mobilenet_engine/fc_wgrad_cos", 1 - cos, 2e-2)
    ok &= report("mobilenet_engine/fc_bgrad", rel_err(eng.g("fc.bias"), ref.fc.bias.grad), 3e-2)
    ok &= report("mobilenet_engine/param_counts", float(eng.trainable_parameters() != 6405) + float(eng.num_parameters() != 2230277), 0.0)
    # through the public API: Trainer.fit on the engine (graph step), loss goes down on a fixed batch; throughput
    from b200ddl import optim
    from b200ddl.train import Trainer
    eng2 = build_model(224, 224, 3, K, dropout=0.0, arch="mobilenetv2", batch_size=64, seed=4)
    tr = Trainer(eng2).compile(optimizer=optim.Adam(0.01), loss="sparse_categorical_crossentropy", metrics=["accuracy"])
    xb = torch.randint(0, 256, (64, 224, 224, 3), device=DEV, dtype=torch.uint8, generator=g)
    yb = torch.randint(0, K, (64,), device=DEV, generator=g)
    hist = tr.fit([(xb, yb)] * 30, steps_per_epoch=30, epochs=2, verbose=0)
    ok &= report("mobilenet_engine/fit_loss_decreases", float(hist.history["loss"][-1] >= hist.history["loss"][0]), 0.0,
                 f"{hist.history['loss'][0]:.3f} -> {hist.history['loss'][-1]:.3f}")
    step = tr.backend.step
    t = time_fn(step.run, iters=10, warmup=3)
    print(f"TIME mobilenet_engine train step batch 64: {t*1e3:.0f} us = {64 / t * 1e3:.0f} images/s", flush=True)
    import time as _t
    refm = build_model(224, 224, 3, K, dropout=0.0, arch="mobilenetv2_torch", seed=4).to(DEV)
    tr2 = Trainer(refm, device=DEV).compile(optimizer=optim.Adam(0.01))
    for _ in range(3):
        tr2.backend.train_batch(xb, yb)
    torch.cuda.synchronize(); t0 = _t.perf_counter()
    for _ in range(10):
        tr2.backend.train_batch(xb, yb)
    torch.cuda.synchronize(); dt = (_t.perf_counter() - t0) / 10
    print(f"TIME mobilenet torch.nn module (eager, fp32) train step batch 64: {dt*1e6:.0f} us = {64 / dt:.0f} images/s", flush=True)
    return ok



def case_umma_probe():
    """Row-shifted SWIZZLE_128B descriptors: which (shift, base_offset) combinations read the right rows?"""
    ext = ops.ext("_b200_probe")
    g = torch.Generator(device=DEV).manual_seed(21)
    T = torch.randn(160, 64, device=DEV, generator=g).to(torch.bfloat16)
    B = torch.randn(64, 64, device=DEV, generator=g).to(torch.bfloat16)
    ok0 = True
    for shift in (0, 1, 2, 3, 7, 8, 9, 30):
        ref = T[shift:shift + 128].float() @ B.float().t()
        res = []
        for bo in (False, True):
            out = ext.umma_probe(T, B, shift, bo)
            torch.cuda.synchronize()
            res.append(rel_err(out, ref))
        print(f"PROBE shift={shift:2d} err(base_offset=0)={res[0]:.3e} err(base_offset=(addr>>7)&7)={res[1]:.3e}", flush=True)
        if shift == 0:
            ok0 &= res[0] < 1e-2
    # second question: 8-row groups at a stride other than 1024 bytes (2-D halo tiles need 1280 = a 10-pixel-wide row)
    T2 = torch.randn(256, 64, device=DEV, generator=g).to(torch.bfloat16)
    for sbo in (1024, 1152, 1280, 1536, 2048):
        step = sbo // 128
        for shift in (0, 1, 11, 22):
            if shift + 15 * step + 8 > 256:
                continue
            rows = torch.cat([torch.arange(shift + gi * step, shift + gi * step + 8, device=DEV) for gi in range(16)])
            ref = T2[rows].float() @ B.float().t()
            out = ext.umma_probe(T2, B, shift, False, sbo)
            torch.cuda.synchronize()
            print(f"PROBE group_stride={sbo:5d} B ({step:2d} rows) shift={shift:2d} err={rel_err(out, ref):.3e}", flush=True)
    return ok0


def case_tma_probe():
    """TMA load pipeline alone (no MMA, no epilogue): time per box load for the shapes the 3x3 convs use or could use."""
    ext = ops.ext("_b200_probe")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    x56 = torch.randn(256, 56, 56, 64, device=DEV).to(torch.bfloat16)
    x28 = torch.randn(512, 28, 28, 64, device=DEV).to(torch.bfloat16)
    wlike = torch.randn(1, 1, 576, 64, device=DEV).to(torch.bfloat16)  # 72 KB, read by every CTA: L2-hot, like a filter

    def run(label, x, rows_2d, box, tap, stages, total_mb=1100.0):
        bw, bh, bn = box
        nbytes = (rows_2d if rows_2d else bw * bh * bn) * 128
        loads = max(8, int(total_mb * 1e6 / nbytes / sms))
        f = lambda: ext.tma_probe(x, rows_2d, bw, bh, bn, tap[0], tap[1], stages, loads, 0)
        for _ in range(3):
            f()
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            f()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) / 5 * 1e3
        tot = loads * sms * nbytes
        print(f"PROBE tma {label:34s} box={nbytes // 128:4d} rows ({nbytes / 1024:5.1f} KB) stages={stages:2d} loads/CTA={loads:5d} "
              f"{us:8.1f} us  {tot / us / 1e6:7.2f} TB/s  {tot / us / 1e3 / sms:6.1f} GB/s/SM  {us * 1e3 / loads:7.1f} ns/load  "
              f"{us * 1e3 / loads / (nbytes // 128):6.2f} ns/row", flush=True)

    run("flat 2-D, 128 rows", x56, 128, (0, 0, 0), (0, 0), 6)
    run("box 56x2x1 (current A tile)", x56, 0, (56, 2, 1), (0, 0), 6)
    run("box 56x2x1 tap(-1,-1)", x56, 0, (56, 2, 1), (-1, -1), 6)
    run("box 56x2x1 tap(+1,+1)", x56, 0, (56, 2, 1), (1, 1), 6)
    run("box 56x2x1 stages 3", x56, 0, (56, 2, 1), (0, 0), 3)
    run("box 56x2x1 stages 12", x56, 0, (56, 2, 1), (0, 0), 12)
    run("box 56x4x1 (halo box)", x56, 0, (56, 4, 1), (0, 0), 4)
    run("box 56x4x1 tap(-1,-1)", x56, 0, (56, 4, 1), (-1, -1), 4)
    run("box 56x4x1 stages 7", x56, 0, (56, 4, 1), (0, 0), 7)
    run("box 8x8x2 (square)", x56, 0, (8, 8, 2), (0, 0), 6)
    run("box 28x4x1 on 28^2", x28, 0, (28, 4, 1), (0, 0), 6)
    run("box 28x6x1 on 28^2 (halo)", x28, 0, (28, 6, 1), (0, 0), 5)
    run("filter-like 64 rows, L2-hot", wlike, 64, (0, 0, 0), (0, 0), 6, total_mb=400.0)
    return True


CASES = {
    "conv_fwd": case_conv_fwd,
    "conv_dgrad": case_conv_dgrad,
    "conv_wgrad": case_conv_wgrad,
    "elementwise": case_elementwise,
    "conv_time": case_conv_time,
    "engine": case_engine,
    "tma_probe": case_tma_probe,
    "engine_serial_wgrad": lambda: case_engine(overlap_wgrad=False, quick=True),
    "stem": case_stem,
    "block_grad": case_block_grad,
    "head": case_head,
    "big_numerics": case_big_numerics,
    "fused_infer": case_fused_infer,
    "mobilenet": case_mobilenet,
    "engine_unfused_block_grad": lambda: case_engine(quick=True, fuse_block_grad=False),
    "umma_probe": case_umma_probe,
}

if __name__ == "__main__":
    torch.backends.cudnn.benchmark = True
    names = sys.argv[1:] or list(CASES)
    allok = True
    for n in names:
        t0 = time.time()
        try:
            ok = CASES[n]()
        except Exception:
            ok = False
            print(f"CASE {n} EXCEPTION\n{traceback.format_exc()}", flush=True)
        allok &= bool(ok)
        print(f"CASE {n} {'PASS' if ok else 'FAIL'} ({time.time() - t0:.1f}s)", flush=True)
    sys.exit(0 if allok else 1)
