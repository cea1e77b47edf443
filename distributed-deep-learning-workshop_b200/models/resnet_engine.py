"""ResNet-50 as a hand-scheduled B200 engine (the TARGET model of BASELINE.json; reference model = C14).

No autograd and no tracing compiler: forward and backward are explicit sequences of our sm_100a kernels over
*static* NHWC bf16 buffers, so the whole training step is one CUDA graph.

  conv            tcgen05/TMEM/TMA implicit GEMM (ops.conv.ConvForward) with the BatchNorm statistics reduced in
                  the epilogue
  BN+ReLU(+add)   one bandwidth-bound pass (bn_apply); backward = reduce pass + apply pass (also emits the masked
                  skip-connection gradient)
  dgrad / wgrad   the same implicit-GEMM kernel with transposed filters / the MN-major wgrad kernel accumulating
                  fp32 straight into the flat gradient buffer the all-reduce consumes
  optimizer       one fused launch over the flat fp32 master / state buffers (see optim.fused)

Parameters live in ONE flat fp32 buffer laid out in *backward completion order*, so gradient buckets become
ready front-to-back and `DistributedOptimizer` can all-reduce bucket k while bucket k+1 is still being computed.
Conv filters use the kernel layout ``[R*S, Cout, Cin]``; `state_dict()` converts to torch's OIHW.

Reference call sites this replaces: `build_model` (P1/03:159-178), `model.fit` inner step (P1/03:353-358).
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional, Tuple

import torch

from .. import ops
from ..ops import conv as C


@dataclass
class ParamSpec:
    name: str
    shape: Tuple[int, ...]
    kind: str  # 'conv' | 'gamma' | 'beta' | 'fc_w' | 'fc_b'
    offset: int = 0
    numel: int = 0


@dataclass
class ConvSpec:
    name: str
    cin: int
    cout: int
    k: int
    stride: int
    pad: int


@dataclass
class BlockSpec:
    name: str
    cin: int
    mid: int
    stride: int
    downsample: bool
    h_in: int
    h_out: int


def _align(n: int, a: int = 64) -> int:
    return (n + a - 1) // a * a


def resnet50_blocks(image_size: int = 224) -> List[BlockSpec]:
    cfg = [(64, 3, 1), (128, 4, 2), (256, 6, 2), (512, 3, 2)]
    blocks = []
    cin = 64
    h = image_size // 4
    for si, (mid, n, stride) in enumerate(cfg):
        for bi in range(n):
            s = stride if bi == 0 else 1
            blocks.append(BlockSpec(f"layer{si + 1}.{bi}", cin, mid, s, bi == 0, h, h // s))
            h //= s
            cin = mid * 4
    return blocks


class ResNet50Engine:
    """Static-shape ResNet-50 training / inference engine for one GPU."""

    arch = "resnet50"

    def __init__(self, batch: int, num_classes: int = 1000, device: Optional[torch.device] = None,
                 image_size: int = 224, dropout: float = 0.0, bn_momentum: float = 0.1, bn_eps: float = 1e-5,
                 seed: int = 0, max_ctas: int = 0, zero_init_residual: bool = True,
                 overlap_wgrad: bool = True, wgrad_smem_budget: int = 0, fuse_bwd_reduce: bool = True,
                 fuse_bn_coeffs: bool = False, fuse_block_grad: Optional[bool] = None,
                 fuse_stem_bwd: Optional[bool] = None):
        if fuse_bn_coeffs:
            raise ValueError("fuse_bn_coeffs was removed: BN coefficients inside the apply kernels measured slower "
                             "(profiles/README.md, section 2.9)")
        if fuse_stem_bwd:
            raise ValueError("fuse_stem_bwd was removed: max-pool backward fused with the stem BN backward measured "
                             "slower (profiles/README.md, R2.4)")
        ops.require_native()
        self.zero_init_residual = zero_init_residual
        # experimental: run every weight-gradient GEMM on a side stream so it overlaps the (DRAM-bound) BatchNorm
        # backward passes of the next layer; needs two dy scratch buffers and event-ordered buffer reuse
        self.overlap_wgrad = overlap_wgrad
        # BatchNorm-backward reductions of bn1/bn2 computed inside the dgrad GEMM that produces their input gradient
        self.fuse_bwd_reduce = fuse_bwd_reduce
        # the gradient merge at every residual-block boundary (main path + skip path, ReLU mask, bn3 reduction) runs in
        # the epilogue of the next block's conv1 dgrad GEMM (conv_igemm kStats = 3); B200DDL_NO_BLOCK_GRAD=1 disables
        self.fuse_block_grad = (os.environ.get("B200DDL_NO_BLOCK_GRAD") != "1") if fuse_block_grad is None else bool(fuse_block_grad)
        self.fuse_stem_bwd = False  # reported by bench.py
        self._fused_reduce = set()
        self._block_fused = set()   # bn3 names whose reduction (and dz) come out of a fused dgrad epilogue
        # inference-only builds (build(training=False)): BatchNorm (running statistics) + ReLU + residual add run in the
        # convolutions' epilogues (conv_igemm kStats = 4) - no BatchNorm pass at all.
        self._infer_fused = False
        self.wgrad_smem_budget = wgrad_smem_budget
        self.aux_streams: List[torch.cuda.Stream] = []
        if image_size % 32:
            raise ValueError("image_size must be a multiple of 32")
        self.batch = int(batch)
        self.num_classes = int(num_classes)
        self.image_size = int(image_size)
        self.dropout = float(dropout)
        self.bn_momentum = bn_momentum
        self.bn_eps = bn_eps
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.max_ctas = int(max_ctas)
        self.seed = seed
        self.blocks = resnet50_blocks(image_size)
        self._e = ops.ext("_b200_ops")
        self._built = False
        self.grad_hook: Optional[Callable[[int, int], None]] = None  # called with flat [lo, hi) when grads are final
        self._step_count = 0
        self._layout_params()
        self._alloc_params(seed)

    # ------------------------------------------------------------------------------------------------ parameters
    def _layout_params(self) -> None:
        specs: List[ParamSpec] = []

        def conv(name, cin, cout, k):
            specs.append(ParamSpec(name + ".weight", (k * k, cout, cin), "conv"))

        def bn(name, c):
            specs.append(ParamSpec(name + ".weight", (c,), "gamma"))
            specs.append(ParamSpec(name + ".bias", (c,), "beta"))

        # backward completion order: fc, blocks reversed (bn3, conv3, bn2, conv2, bn1, [bn_ds, conv_ds], conv1), stem.
        # The FC filter is stored with its class dimension padded to a GEMM-friendly size (zero rows: zero gradient,
        # so they stay zero under SGD / Adam / Adadelta); state_dict() exposes the real [num_classes, 2048] slice.
        self.classes_padded = 64 if self.num_classes <= 64 else _align(self.num_classes, 128)
        specs.append(ParamSpec("fc.weight", (self.classes_padded, 2048), "fc_w"))
        specs.append(ParamSpec("fc.bias", (self.num_classes,), "fc_b"))
        for b in reversed(self.blocks):
            bn(b.name + ".bn3", b.mid * 4)
            conv(b.name + ".conv3", b.mid, b.mid * 4, 1)
            bn(b.name + ".bn2", b.mid)
            conv(b.name + ".conv2", b.mid, b.mid, 3)
            bn(b.name + ".bn1", b.mid)
            if b.downsample:
                bn(b.name + ".downsample.1", b.mid * 4)
                conv(b.name + ".downsample.0", b.cin, b.mid * 4, 1)
            conv(b.name + ".conv1", b.cin, b.mid, 1)
        bn("bn1", 64)
        specs.append(ParamSpec("conv1.weight", (49, 64, 3), "conv"))
        off = 0
        for s in specs:
            s.numel = int(math.prod(s.shape))
            s.offset = off
            off += _align(s.numel)
        self.param_specs = specs
        self.spec = {s.name: s for s in specs}
        self.flat_numel = off

    def _alloc_params(self, seed: int) -> None:
        dev = self.device
        self.params = torch.zeros(self.flat_numel, device=dev, dtype=torch.float32)
        self.w16 = torch.zeros(self.flat_numel, device=dev, dtype=torch.bfloat16)
        self.grads: Optional[torch.Tensor] = None  # bound later (may be symmetric memory)
        g = torch.Generator(device="cpu").manual_seed(seed)
        for s in self.param_specs:
            v = self.params[s.offset:s.offset + s.numel].view(s.shape)
            if s.kind == "conv":
                taps, cout, cin = s.shape
                std = math.sqrt(2.0 / (cout * taps))  # kaiming normal, fan_out (torchvision)
                v.copy_(torch.randn(s.shape, generator=g) * std)
            elif s.kind == "gamma":
                # zero-init the last BN of every residual branch (Goyal et al., cited by the reference P1/03:315)
                v.fill_(0.0 if (self.zero_init_residual and s.name.endswith("bn3.weight")) else 1.0)
            elif s.kind == "fc_w":
                bound = 1.0 / math.sqrt(2048)
                v[:self.num_classes].copy_((torch.rand((self.num_classes, 2048), generator=g) * 2 - 1) * bound)
            elif s.kind == "fc_b":
                bound = 1.0 / math.sqrt(2048)
                v.copy_((torch.rand(s.shape, generator=g) * 2 - 1) * bound)
        # running statistics (not optimised): one flat buffer, mean then var per BN
        self.bn_names = [s.name[:-len(".weight")] for s in self.param_specs if s.kind == "gamma"]
        self.bn_channels = {n: self.spec[n + ".weight"].numel for n in self.bn_names}
        tot = sum(self.bn_channels.values())
        self.running = torch.zeros(2 * tot, device=dev)
        self.running_mean: Dict[str, torch.Tensor] = {}
        self.running_var: Dict[str, torch.Tensor] = {}
        o = 0
        for n in self.bn_names:
            c = self.bn_channels[n]
            self.running_mean[n] = self.running[o:o + c]
            self.running_var[n] = self.running[tot + o:tot + o + c]
            o += c
        self.running[tot:].fill_(1.0)
        self.sync_weights()

    def p(self, name: str) -> torch.Tensor:
        s = self.spec[name]
        return self.params[s.offset:s.offset + s.numel].view(s.shape)

    def g(self, name: str) -> torch.Tensor:
        s = self.spec[name]
        return self.grads[s.offset:s.offset + s.numel].view(s.shape)

    def w16v(self, name: str) -> torch.Tensor:
        s = self.spec[name]
        return self.w16[s.offset:s.offset + s.numel].view(s.shape)

    def sync_weights(self) -> None:
        """Refresh every bf16 working copy from the fp32 master (after an optimizer step or a weight load)."""
        self._e.cast_bf16(self.params, self.w16)
        if self._built:
            self.refresh_derived_weights()

    def refresh_derived_weights(self) -> None:
        """bf16 copies in layouts other than the master's: dgrad filters (one batched kernel + the few stride-2
        tap subsets) and the packed stem filter."""
        if getattr(self, "_wd_total", 0) > 0:
            self._e.weight_prep_batched(self.params, self._wd16, self._wd_table, self._wd_tiles)
        self._refresh_stem_weight()
        if self._infer_fused:
            self._refresh_eval_affine()

    def _refresh_eval_affine(self) -> None:
        """scale / shift of every BatchNorm from its running statistics (inference epilogues read them)."""
        for bn in self.bn_names:
            self._bn_fwd(bn, 1.0, False)

    def _refresh_stem_weight(self) -> None:
        self._e.pack_stem_weight(self.p("conv1.weight"), self._stem_w16)

    # ------------------------------------------------------------------------------------------------ build
    def bind_grad_buffer(self, grads: Optional[torch.Tensor] = None) -> None:
        if grads is None:
            grads = torch.zeros(self.flat_numel, device=self.device, dtype=torch.float32)
        assert grads.numel() >= self.flat_numel and grads.dtype == torch.float32
        self.grads = grads

    def build(self, training: bool = True) -> "ResNet50Engine":
        """Allocate activations / scratch and encode every TMA descriptor (once; buffers are static)."""
        if self._built:
            if not (training and not self._training_built):
                return self
            # built for inference (fused epilogues, no backward buffers) and now asked to train: build again
            self._built = False
            self._fused_reduce.clear()
            self._block_fused.clear()
        if self.grads is None and training:
            self.bind_grad_buffer()
        dev, N, e = self.device, self.batch, self._e
        bf = dict(device=dev, dtype=torch.bfloat16)
        f32 = dict(device=dev, dtype=torch.float32)
        S = self.image_size
        self.x_u8 = torch.zeros(N, S, S, 3, device=dev, dtype=torch.uint8)
        self.labels = torch.zeros(N, device=dev, dtype=torch.int64)
        self.stats = torch.zeros(2, **f32)          # [sum loss, correct]
        self.logits = torch.zeros(N, self.num_classes, **f32)  # fp32 logits (+bias) for predict(); written by the CE kernel
        self.loss_rows = torch.zeros(N, **f32)

        # BN work buffers (per BN): sum, sqsum, mean, invstd, scale, shift, sum_dz, sum_dzy, cA, cB, cC
        # The four accumulators of ALL layers live in two contiguous buffers so that one memset per pass zeroes them.
        self.bnw: Dict[str, Dict[str, torch.Tensor]] = {}
        total_c = sum(self.bn_channels[n] for n in self.bn_names)
        self._bn_fwd_sums = torch.zeros(2, total_c, **f32)   # [sum | sqsum] filled by the conv epilogues
        self._bn_bwd_sums = torch.zeros(2, total_c, **f32)   # [sum_dz | sum_dzy] filled by reduce kernels / dgrad epilogues
        off = 0
        for n in self.bn_names:
            c = self.bn_channels[n]
            buf = torch.zeros(7, c, **f32)
            keys = ["mean", "invstd", "scale", "shift", "cA", "cB", "cC"]
            self.bnw[n] = {k: buf[i] for i, k in enumerate(keys)}
            self.bnw[n]["sum"] = self._bn_fwd_sums[0, off:off + c]
            self.bnw[n]["sqsum"] = self._bn_fwd_sums[1, off:off + c]
            self.bnw[n]["sum_dz"] = self._bn_bwd_sums[0, off:off + c]
            self.bnw[n]["sum_dzy"] = self._bn_bwd_sums[1, off:off + c]
            off += c

        H0 = S // 2
        self.y0 = torch.zeros(N, H0, H0, 64, **bf)
        self.p0 = torch.zeros(N, H0 // 2, H0 // 2, 64, **bf)
        self.pool_idx = torch.zeros(N, H0 // 2, H0 // 2, 64, device=dev, dtype=torch.uint8)
        w0 = self.bnw["bn1"]
        self._stem_w16 = torch.zeros(64, 192, **bf)
        self._stem_fwd = C.StemForward(self.x_u8, self._stem_w16, self.y0, w0["sum"], w0["sqsum"], max_ctas=self.max_ctas)
        self._refresh_stem_weight()

        max_act = N * (S // 4) * (S // 4) * 256
        max_act = max(max_act, N * H0 * H0 * 64)
        if training:
            self._scr = {k: torch.zeros(max_act, **bf) for k in ("dy", "dyB", "da", "dds", "dzA", "dzB")}
            # the downsample branch runs between bn1's backward and conv1's (whose dy sits in "dy"): always its own buffer
            self._dy_key = {"conv3": "dy", "conv2": "dyB" if self.overlap_wgrad else "dy", "conv1": "dy",
                            "downsample.0": "dyB"}
            self._dy_reader: Dict[str, torch.cuda.Event] = {}
            if self.overlap_wgrad:
                self._wg_stream = torch.cuda.Stream(device=dev)
                self.aux_streams = [self._wg_stream]

        # bf16 dgrad copies ([tap][Cin][Cout]) of EVERY filter (stride-1 layers whole, stride-2 layers per output-parity
        # tap subset, the FC matrix) live in one flat buffer refreshed by ONE kernel (weight_prep_batched).
        self._wd_table_rows = []
        self._wd_slices: Dict[str, List[Tuple[int, int]]] = {}   # conv name -> [(offset, numel)] per dgrad part
        wd_total = 0
        wd_tiles = 0   # 64 (co) x 32 (ci) transpose tiles, the unit of work of weight_prep_batched

        def add_dgrad_weights(full: str, parts: List[List[int]]):
            nonlocal wd_total, wd_tiles
            sp = self.spec[full + ".weight"]
            taps, cout, cin = sp.shape if len(sp.shape) == 3 else (1, sp.shape[0], sp.shape[1])
            out = []
            for idx in parts:
                start = wd_total
                i = 0
                while i < len(idx):  # one table row per run of consecutive taps
                    j = i
                    while j + 1 < len(idx) and idx[j + 1] == idx[j] + 1:
                        j += 1
                    n = j - i + 1
                    assert cout % 64 == 0 and cin % 32 == 0
                    self._wd_table_rows.append([sp.offset + idx[i] * cout * cin, wd_total, n, cout, cin, wd_tiles])
                    wd_total += n * cout * cin
                    wd_tiles += n * (cout // 64) * (cin // 32)
                    i = j + 1
                out.append((start, wd_total - start))
            self._wd_slices[full] = out

        fuse_bg = self.fuse_block_grad and training
        if training:
            add_dgrad_weights("fc", [[0]])
            for bi, b in enumerate(self.blocks):
                for cname, k, stride in (("conv1", 1, 1), ("conv2", 3, b.stride), ("conv3", 1, 1),
                                         ("downsample.0", 1, b.stride)):
                    if cname == "downsample.0" and not b.downsample:
                        continue
                    if cname == "downsample.0" and stride == 2 and fuse_bg and bi > 0:
                        parts = [[0]]  # compact dgrad: a dense 1x1 GEMM on the strided grid
                    else:
                        parts = C.ConvDgrad.part_taps(k, k, stride, (k - 1) // 2)
                    add_dgrad_weights(b.name + "." + cname, parts)
            assert len(self._wd_table_rows) <= 128
            self._wd16 = torch.zeros(max(wd_total, 8), **bf)
            self._wd_total = wd_total
            self._wd_tiles = wd_tiles
            self._wd_table = torch.tensor(self._wd_table_rows, device=dev, dtype=torch.int64).view(-1, 6)

        def wd_views(full: str) -> List[torch.Tensor]:
            return [self._wd16[o:o + n] for o, n in self._wd_slices[full]]

        self.act: Dict[str, torch.Tensor] = {}
        self._fwd: Dict[str, C.ConvForward] = {}
        self._dg: Dict[str, C.ConvDgrad] = {}
        self._wg: Dict[str, C.ConvWgrad] = {}
        self._dgrads: List[C.ConvDgrad] = []
        mc = self.max_ctas

        def scr(key, shape):
            n = int(math.prod(shape))
            return self._scr[key][:n].view(shape)

        dz_keys = ["dzA", "dzB"]
        x_in = self.p0
        self._infer_fused = not training
        for bi, b in enumerate(self.blocks if self._infer_fused else []):
            # inference: every convolution writes its block activation directly (folded BN + ReLU [+ residual] epilogue)
            Hi, Ho, mid, cout = b.h_in, b.h_out, b.mid, b.mid * 4
            A, n = self.act, b.name
            A[n + ".a1"] = torch.zeros(N, Hi, Hi, mid, **bf)
            A[n + ".a2"] = torch.zeros(N, Ho, Ho, mid, **bf)
            A[n + ".out"] = torch.zeros(N, Ho, Ho, cout, **bf)

            def w2d(full):
                w = self.w16v(full + ".weight")
                return w.view(w.shape[0] * w.shape[1], w.shape[2])

            def aff(bn, act, res=None):
                return (self.bnw[n + "." + bn]["scale"], self.bnw[n + "." + bn]["shift"], act, res)

            self._fwd[n + ".conv1"] = C.ConvForward(x_in, w2d(n + ".conv1"), A[n + ".a1"], 1, 1, 1, 0, None, None, mc,
                                                    epilogue=aff("bn1", "relu"))
            self._fwd[n + ".conv2"] = C.ConvForward(A[n + ".a1"], w2d(n + ".conv2"), A[n + ".a2"], 3, 3, b.stride, 1, None,
                                                    None, mc, epilogue=aff("bn2", "relu"))
            res = x_in
            if b.downsample:
                A[n + ".yd"] = torch.zeros(N, Ho, Ho, cout, **bf)
                self._fwd[n + ".downsample.0"] = C.ConvForward(x_in, w2d(n + ".downsample.0"), A[n + ".yd"], 1, 1, b.stride,
                                                               0, None, None, mc, epilogue=aff("downsample.1", "none"))
                res = A[n + ".yd"]
            self._fwd[n + ".conv3"] = C.ConvForward(A[n + ".a2"], w2d(n + ".conv3"), A[n + ".out"], 1, 1, 1, 0, None, None,
                                                    mc, epilogue=aff("bn3", "relu", res))
            x_in = A[n + ".out"]
        for bi, b in enumerate([] if self._infer_fused else self.blocks):
            Hi, Ho, mid, cout = b.h_in, b.h_out, b.mid, b.mid * 4
            A = self.act
            A[b.name + ".y1"] = torch.zeros(N, Hi, Hi, mid, **bf)
            A[b.name + ".a1"] = torch.zeros(N, Hi, Hi, mid, **bf)
            A[b.name + ".y2"] = torch.zeros(N, Ho, Ho, mid, **bf)
            A[b.name + ".a2"] = torch.zeros(N, Ho, Ho, mid, **bf)
            A[b.name + ".y3"] = torch.zeros(N, Ho, Ho, cout, **bf)
            A[b.name + ".out"] = torch.zeros(N, Ho, Ho, cout, **bf)
            if training:  # 1 bit per element ReLU mask of the block output (read by the backward pass)
                A[b.name + ".mask"] = torch.zeros(N * Ho * Ho * cout // 8, device=dev, dtype=torch.uint8)
            if b.downsample:
                A[b.name + ".yd"] = torch.zeros(N, Ho, Ho, cout, **bf)
            convs = [("conv1", x_in, "y1", "bn1", 1, 1, 0), ("conv2", A[b.name + ".a1"], "y2", "bn2", 3, b.stride, 1),
                     ("conv3", A[b.name + ".a2"], "y3", "bn3", 1, 1, 0)]
            if b.downsample:
                convs.append(("downsample.0", x_in, "yd", "downsample.1", 1, b.stride, 0))
            for cname, xin, yk, bnk, k, stride, pad in convs:
                full = b.name + "." + cname
                w = self.w16v(full + ".weight")
                w2d = w.view(w.shape[0] * w.shape[1], w.shape[2])
                bw_ = self.bnw[b.name + "." + bnk]
                y = A[b.name + "." + yk]
                self._fwd[full] = C.ConvForward(xin, w2d, y, k, k, stride, pad, bw_["sum"], bw_["sqsum"], mc)
                if training:
                    dy = scr(self._dy_key[cname], y.shape)
                    gw = self.g(full + ".weight")
                    self._wg[full] = C.ConvWgrad(dy, xin, gw.view(gw.shape[0] * gw.shape[1], gw.shape[2]), k, k,
                                                 stride, pad, 0, mc, self.wgrad_smem_budget)
                    bwd_stats = None
                    block_grad = None
                    d_stride = stride
                    if cname == "downsample.0":
                        if stride == 2 and fuse_bg and bi > 0:
                            # compact gradient on the strided grid; the fused conv1 epilogue scatters it on the fly
                            dx = scr("dds", (N, Ho, Ho, b.cin))
                            d_stride = 1
                        else:
                            dx = scr("dds", xin.shape)
                    elif cname == "conv1" and fuse_bg and bi > 0:
                        # dx = complete masked gradient dz of the PREVIOUS block's output (+ its bn3 reduction)
                        pb = self.blocks[bi - 1]
                        dx = scr(dz_keys[(bi - 1) % 2], xin.shape)
                        skip = scr("dds", (N, Ho, Ho, b.cin) if b.stride == 2 else xin.shape) if b.downsample \
                            else scr(dz_keys[bi % 2], xin.shape)
                        pw = self.bnw[pb.name + ".bn3"]
                        block_grad = (skip, A[pb.name + ".mask"], A[pb.name + ".y3"], pw["sum_dz"], pw["sum_dzy"])
                        self._block_fused.add(pb.name + ".bn3")
                    else:
                        dx = scr("da", xin.shape)
                    if self.fuse_bwd_reduce and stride == 1 and cname in ("conv2", "conv3"):
                        # dx is the gradient of a1 (conv2) / a2 (conv3): fuse the reduction of bn1 / bn2
                        pbn = "bn1" if cname == "conv2" else "bn2"
                        pw = self.bnw[b.name + "." + pbn]
                        py = A[b.name + (".y1" if cname == "conv2" else ".y2")]
                        bwd_stats = (py, pw["scale"], pw["shift"], pw["sum_dz"], pw["sum_dzy"])
                        self._fused_reduce.add(b.name + "." + pbn)
                    dgr = C.ConvDgrad(dy, self.p(full + ".weight"), dx, k, k, d_stride, pad, mc, wbufs=wd_views(full),
                                      bwd_stats=bwd_stats, block_grad=block_grad)
                    self._dg[full] = dgr
                    self._dgrads.append(dgr)
            x_in = A[b.name + ".out"]
        self.feat = x_in  # [N, 7, 7, 2048]
        self.pooled = torch.zeros(N, 2048, **bf)
        # classifier head on the same tcgen05 kernels: a 1x1 "convolution" over a 1x1 image (reference Dense, P1/02:175)
        ncp = self.classes_padded
        self.logits16 = torch.zeros(N, ncp, **bf)
        self._fc_fwd = C.ConvForward(self.pooled.view(N, 1, 1, 2048), self.w16v("fc.weight"), self.logits16.view(N, 1, 1, ncp),
                                     1, 1, 1, 0, None, None, mc)
        if training:
            self.dlogits16 = torch.zeros(N, ncp, **bf)
            self.dpooled = torch.zeros(N, 2048, **bf)
            self._fc_wg = C.ConvWgrad(self.dlogits16.view(N, 1, 1, ncp), self.pooled.view(N, 1, 1, 2048),
                                      self.g("fc.weight"), 1, 1, 1, 0, 0, mc, 0)
            self._fc_dg = C.ConvDgrad(self.dlogits16.view(N, 1, 1, ncp), self.p("fc.weight").view(1, ncp, 2048),
                                      self.dpooled.view(N, 1, 1, 2048), 1, 1, 1, 0, mc, wbufs=wd_views("fc"))
            dy0 = self._scr["dzA"][:self.y0.numel()].view(self.y0.shape)
            self._stem_wg = C.StemWgrad(self.x_u8, dy0, self.g("conv1.weight").view(-1), max_ctas=self.max_ctas)
        self._training_built = training
        self._built = True
        self.sync_weights()
        return self

    # ------------------------------------------------------------------------------------------------ forward
    def _bn_fwd(self, bn: str, count: float, training: bool) -> Dict[str, torch.Tensor]:
        w = self.bnw[bn]
        self._e.bn_finalize(w["sum"], w["sqsum"], float(count), self.p(bn + ".weight"), self.p(bn + ".bias"),
                            self.running_mean[bn], self.running_var[bn], self.bn_momentum, self.bn_eps, w["mean"],
                            w["invstd"], w["scale"], w["shift"], training)
        return w

    def _bn_apply(self, bn: str, count: float, training: bool, y, out, res=None, res_bn: Optional[str] = None,
                  mask=None) -> None:
        """out = relu(BN(y) [+ res | + BN_res(res)])."""
        e = self._e
        w = self._bn_fwd(bn, count, training)
        if res_bn is not None:
            wd = self._bn_fwd(res_bn, count, training)
            e.bn_apply(y, w["scale"], w["shift"], res, wd["scale"], wd["shift"], out, True, mask)
        else:
            e.bn_apply(y, w["scale"], w["shift"], res, None, None, out, True, mask)

    def forward(self, training: bool = True) -> None:
        """x_u8 / labels (static inputs) -> logits, loss stats.  All launches go to the current stream."""
        e, N, A = self._e, self.batch, self.act
        w0 = self.bnw["bn1"]
        # 7x7/2 stem on the tensor cores straight from the uint8 batch (normalisation + BN statistics fused)
        self._stem_fwd.run()
        cnt0 = N * self.y0.shape[1] * self.y0.shape[2]
        self._bn_fwd("bn1", cnt0, training)
        # BN + ReLU + 3x3/2 max-pool in one pass (the 112x112 activation is never written)
        e.bn_relu_maxpool_fwd(self.y0, w0["scale"], w0["shift"], self.p0, self.pool_idx)
        x_in = self.p0
        if self._infer_fused and not training:
            for b in self.blocks:
                n = b.name
                self._fwd[n + ".conv1"].run()
                self._fwd[n + ".conv2"].run()
                if b.downsample:
                    self._fwd[n + ".downsample.0"].run()
                self._fwd[n + ".conv3"].run()
        for b in ([] if (self._infer_fused and not training) else self.blocks):
            n = b.name
            cnt_in = N * b.h_in * b.h_in
            cnt_out = N * b.h_out * b.h_out
            self._fwd[n + ".conv1"].run()
            self._bn_apply(n + ".bn1", cnt_in, training, A[n + ".y1"], A[n + ".a1"])
            self._fwd[n + ".conv2"].run()
            self._bn_apply(n + ".bn2", cnt_out, training, A[n + ".y2"], A[n + ".a2"])
            self._fwd[n + ".conv3"].run()
            mask = A.get(n + ".mask") if training else None
            if b.downsample:
                self._fwd[n + ".downsample.0"].run()
                self._bn_apply(n + ".bn3", cnt_out, training, A[n + ".y3"], A[n + ".out"], A[n + ".yd"],
                               n + ".downsample.1", mask)
            else:
                self._bn_apply(n + ".bn3", cnt_out, training, A[n + ".y3"], A[n + ".out"], x_in, None, mask)
            x_in = A[n + ".out"]
        drop = self.dropout if training else 0.0
        self._drop_seed = self.seed * 1000003 + self._step_count
        e.gap_fwd(self.feat, self.pooled, drop, self._drop_seed)
        self._fc_fwd.run()  # bf16 logits (class dimension padded) on the tcgen05 GEMM
        e.zero_(self.stats)
        # + bias, softmax cross-entropy, accuracy, bf16 dlogits (padded columns zero) in one kernel
        e.softmax_ce_head(self.logits16, self.p("fc.bias"), self.labels, self.logits,
                          self.dlogits16 if training else None, self.loss_rows, self.stats, 1.0 / N)

    # ------------------------------------------------------------------------------------------------ backward
    def _ready(self, *names: str) -> None:
        if self.grad_hook is None:
            return
        lo = min(self.spec[n].offset for n in names)
        hi = max(self.spec[n].offset + _align(self.spec[n].numel) for n in names)
        self.grad_hook(lo, hi)

    def _bn_bwd(self, bn: str, mode: int, g1, g2, out, y, dy, dz, count: float) -> None:
        """BatchNorm(+ReLU) backward = reduce pass + apply pass.

        mode 1: block-final BN: dz = (g1 + g2) * (out > 0) is stored (it is also the skip-connection gradient);
        mode 2: BN + ReLU without residual: the mask is recomputed from y (no read of the activation);
        mode 3: BN without ReLU (downsample branch): dz = g1."""
        e, w = self._e, self.bnw[bn]
        if mode == 1:
            # `out` is the 1-bit ReLU mask written by the forward pass (reduce mode 4).  When the next block's conv1
            # dgrad carried the block-gradient epilogue, dz and both sums already exist (g1 is None).
            if g1 is not None:
                e.bn_bwd_reduce(4, g1, g2, out, y, None, None, dz, w["sum_dz"], w["sum_dzy"])
        elif mode == 2:
            if bn not in self._fused_reduce:  # otherwise the dgrad GEMM that produced g1 already accumulated the sums
                e.bn_bwd_reduce(2, g1, None, None, y, w["scale"], w["shift"], None, w["sum_dz"], w["sum_dzy"])
        else:
            e.bn_bwd_reduce(3, g1, None, None, y, None, None, None, w["sum_dz"], w["sum_dzy"])
        src = dz if mode == 1 else g1
        sc, sh = (w["scale"], w["shift"]) if mode == 2 else (None, None)
        e.bn_bwd_coeffs(w["sum_dz"], w["sum_dzy"], self.p(bn + ".weight"), w["mean"], w["invstd"], float(count),
                        self.g(bn + ".weight"), self.g(bn + ".bias"), w["cA"], w["cB"], w["cC"])
        e.bn_bwd_apply(src, y, sc, sh, w["cA"], w["cB"], w["cC"], dy)
        self._ready(bn + ".weight", bn + ".bias")

    def _dy_buf(self, cname: str, shape) -> torch.Tensor:
        """Scratch view that will receive dy of `cname`; waits for the side-stream wgrad that last read the buffer."""
        key = self._dy_key[cname]
        if self.overlap_wgrad and key in self._dy_reader:
            torch.cuda.current_stream().wait_event(self._dy_reader.pop(key))
        return self._scr[key][:int(math.prod(shape))].view(shape)

    def _conv_bwd(self, full: str, cname: str) -> None:
        """dgrad on the compute stream; wgrad either in line or on the side stream once dgrad has been issued."""
        if not self.overlap_wgrad:
            self._wg[full].run()
            self._dg[full].run()
            # only after every reader of this layer's weights has been enqueued: with fused_update the bucket kernel
            # launched from the hook rewrites them
            self._ready(full + ".weight")
            return
        self._dg[full].run()
        ev = torch.cuda.Event()
        ev.record()
        self._wg_stream.wait_event(ev)
        with torch.cuda.stream(self._wg_stream):
            self._wg[full].run()
            done = torch.cuda.Event()
            done.record()
        self._dy_reader[self._dy_key[cname]] = done
        self._ready(full + ".weight")

    def backward(self) -> None:
        """dlogits -> every parameter gradient (fp32, written into the flat gradient buffer)."""
        e, N, A = self._e, self.batch, self.act
        e.zero_(self.grads)  # wgrad accumulates with atomics
        # classifier head: wgrad + dgrad on the tcgen05 GEMMs, bias gradient = column sums of dlogits
        self._fc_wg.run()
        e.fc_bias_grad(self.dlogits16, self.g("fc.bias"))
        self._fc_dg.run()
        self._ready("fc.weight", "fc.bias")
        drop = self.dropout
        gshape = self.feat.shape
        g1 = self._scr["da"][:self.feat.numel()].view(gshape)
        e.gap_bwd(self.dpooled, g1, drop, self._drop_seed)
        g2 = None
        dz_keys = ["dzA", "dzB"]
        for bi in range(len(self.blocks) - 1, -1, -1):
            b = self.blocks[bi]
            n = b.name
            x_in = A[self.blocks[bi - 1].name + ".out"] if bi > 0 else self.p0
            cnt_in = N * b.h_in * b.h_in
            cnt_out = N * b.h_out * b.h_out
            y3 = A[n + ".y3"]
            dy3 = self._dy_buf("conv3", y3.shape)
            dz = self._scr[dz_keys[bi % 2]][:y3.numel()].view(y3.shape)
            if (n + ".bn3") in self._block_fused:
                # dz and the bn3 sums were produced by the epilogue of the next block's conv1 dgrad
                self._bn_bwd(n + ".bn3", 1, None, None, A[n + ".mask"], y3, dy3, dz, cnt_out)
            else:
                self._bn_bwd(n + ".bn3", 1, g1, g2, A[n + ".mask"], y3, dy3, dz, cnt_out)
            self._conv_bwd(n + ".conv3", "conv3")  # dgrad -> da (a2-shaped)
            da2 = self._scr["da"][:A[n + ".a2"].numel()].view(A[n + ".a2"].shape)
            y2 = A[n + ".y2"]
            dy2 = self._dy_buf("conv2", y2.shape)
            self._bn_bwd(n + ".bn2", 2, da2, None, None, y2, dy2, None, cnt_out)
            self._conv_bwd(n + ".conv2", "conv2")  # dgrad -> da (a1-shaped)
            y1, a1 = A[n + ".y1"], A[n + ".a1"]
            da1 = self._scr["da"][:a1.numel()].view(a1.shape)
            dy1 = self._dy_buf("conv1", y1.shape)
            self._bn_bwd(n + ".bn1", 2, da1, None, None, y1, dy1, None, cnt_in)
            if b.downsample:
                # the downsample branch receives the same masked gradient dz; its BN has no ReLU.  It runs BEFORE the
                # conv1 dgrad, whose epilogue may consume its output as the skip gradient of the previous block.
                yd = A[n + ".yd"]
                dyd = self._dy_buf("downsample.0", yd.shape)
                self._bn_bwd(n + ".downsample.1", 3, dz, None, None, yd, dyd, None, cnt_out)
                self._conv_bwd(n + ".downsample.0", "downsample.0")  # dgrad -> dds (x_in-shaped, or compact)
                g2 = self._dg[n + ".downsample.0"].dx
            else:
                g2 = dz
            # dgrad -> main-path gradient of the block input, or (fused) the previous block's complete dz
            self._conv_bwd(n + ".conv1", "conv1")
            g1 = self._dg[n + ".conv1"].dx
        # stem: g1 (main path of layer1.0) + g2 (its projection shortcut) flow through max-pool, ReLU and bn1
        dy0 = self._scr["dzA"][:self.y0.numel()].view(self.y0.shape)
        cnt0 = N * self.y0.shape[1] * self.y0.shape[2]
        da0 = self._dy_buf("conv3", self.y0.shape)  # reuses the (by now idle) "dy" scratch
        e.maxpool_bwd(self.pool_idx, g1, g2, da0)
        self._bn_bwd("bn1", 2, da0, None, None, self.y0, dy0, None, cnt0)
        self._stem_wg.run()
        self._ready("conv1.weight")
        if self.overlap_wgrad:
            torch.cuda.current_stream().wait_stream(self._wg_stream)
            self._dy_reader.clear()

    # ------------------------------------------------------------------------------------------------ utilities
    def set_input(self, x_u8: torch.Tensor, labels: Optional[torch.Tensor] = None) -> None:
        """Copy a batch into the static input buffers.  Images whose spatial size differs from the engine's are resized
        ON THE GPU (bilinear, half-pixel centres like `tf.image.resize` - the reference's preprocess, P1/03:182-189):
        the batch goes to a device staging buffer of its own size and `resize_bilinear_u8` writes the engine input."""
        if x_u8.dim() == 4 and tuple(x_u8.shape[1:3]) != (self.image_size, self.image_size):
            if x_u8.shape[0] != self.batch or x_u8.shape[3] != 3 or x_u8.dtype != torch.uint8:
                raise ValueError(f"set_input: expected uint8 [{self.batch}, H, W, 3], got {tuple(x_u8.shape)} {x_u8.dtype}")
            key = tuple(x_u8.shape)
            stage = getattr(self, "_resize_stage", {}).get(key)
            if stage is None:
                if not hasattr(self, "_resize_stage"):
                    self._resize_stage = {}
                stage = self._resize_stage[key] = torch.empty(key, device=self.device, dtype=torch.uint8)
            stage.copy_(x_u8, non_blocking=True)
            self._e.resize_bilinear_u8(stage, self.x_u8)
        else:
            self.x_u8.copy_(x_u8.view(self.x_u8.shape), non_blocking=True)
        if labels is not None:
            self.labels.copy_(labels, non_blocking=True)

    def loss_and_acc(self) -> Tuple[float, float]:
        s = self.stats.tolist()
        return s[0] / self.batch, s[1] / self.batch

    def state_dict(self) -> Dict[str, torch.Tensor]:
        """torch / torchvision-compatible names and layouts (conv OIHW)."""
        sd = {}
        for s in self.param_specs:
            v = self.p(s.name).detach().clone()
            if s.kind == "conv":
                k = int(round(math.sqrt(s.shape[0])))
                v = C.weight_from_kernel_layout(v, k, k)
            elif s.kind == "fc_w":
                v = v[:self.num_classes].contiguous()  # drop the zero padding rows
            sd[s.name] = v.cpu()
        for n in self.bn_names:
            sd[n + ".running_mean"] = self.running_mean[n].detach().clone().cpu()
            sd[n + ".running_var"] = self.running_var[n].detach().clone().cpu()
        return sd

    def load_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        for s in self.param_specs:
            v = sd[s.name].to(self.device, torch.float32)
            if s.kind == "conv":
                v = C.weight_to_kernel_layout(v)
            if s.kind == "fc_w":
                self.p(s.name).zero_()
                self.p(s.name)[:self.num_classes].copy_(v)
                continue
            self.p(s.name).copy_(v)
        for n in self.bn_names:
            if n + ".running_mean" in sd:
                self.running_mean[n].copy_(sd[n + ".running_mean"])
                self.running_var[n].copy_(sd[n + ".running_var"])
        self.sync_weights()

    def num_parameters(self) -> int:
        return sum(s.numel for s in self.param_specs) - (self.classes_padded - self.num_classes) * 2048


class EngineTrainStep:
    """forward + backward + (distributed) optimizer update of a `ResNet50Engine`, captured as ONE CUDA graph.

    ``optimizer`` is a `b200ddl.optim` flat optimizer or a `b200ddl.parallel.DistributedOptimizer` around one.
    Usage per step::

        step.load(x_u8, labels)   # H2D / D2D into the static input buffers (outside the graph)
        step.run()                # graph replay (or eager launches when use_graph=False)
        loss, acc = step.result() # D2H of the two fp32 statistics
    """

    def __init__(self, engine: ResNet50Engine, optimizer, use_graph: bool = True, warmup_steps: int = 2):
        from ..parallel import core as _core
        from ..utils.timeline import timeline_from_env

        self.engine = engine
        self.optimizer = optimizer
        self.timeline = timeline_from_env(_core.rank())  # B200DDL_TIMELINE=trace.json (HOROVOD_TIMELINE equivalent)
        if self.timeline is not None:
            use_graph = False  # CUDA-event timing cannot be captured into a graph
        self.use_graph = use_graph
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self._dist = hasattr(optimizer, "on_grads_ready")
        if self._dist:
            optimizer.timeline = self.timeline
            optimizer.extra_wait_streams = engine.aux_streams if engine.aux_streams else []
        e = engine
        ranges = [(s.offset, s.offset + _align(s.numel)) for s in e.param_specs]
        if self._dist:
            grads = optimizer.allocate_grads(e.flat_numel, e.device)
            e.bind_grad_buffer(grads)
            if getattr(optimizer, "fused_update", False):
                # fused all-reduce + SGD: master weights and the bf16 copy move to symmetric/multicast memory
                e.params, e.w16 = optimizer.allocate_weights(e.params, e.w16)
            optimizer.attach(e.params, ranges, e.w16, grads)
            e.grad_hook = optimizer.on_grads_ready
        else:
            e.bind_grad_buffer()
            optimizer.attach(e.params, e.grads, e.w16)
        e.build(training=True)
        if self._dist:
            optimizer.extra_wait_streams = list(e.aux_streams)
        self._warmup_steps = warmup_steps
        self._host_stats = torch.zeros(2, dtype=torch.float32).pin_memory()
        self.steps = 0
        self._captured = False

    # one full step as a launch sequence on the current stream
    def _launch(self) -> None:
        e, opt, tl = self.engine, self.optimizer, self.timeline
        if self._dist:
            opt.start_backward()
        if tl is None:
            e.forward(training=True)
            e.backward()
            opt.step()  # distributed: waits for the comm stream first
            e.refresh_derived_weights()
            return
        with tl.device_span("forward", "step"):
            e.forward(training=True)
        with tl.device_span("backward", "step"):
            e.backward()
        with tl.device_span("allreduce_wait+optimizer", "step"):
            opt.step()
        with tl.device_span("weight_relayout", "step"):
            e.refresh_derived_weights()

    def dump_timeline(self) -> Optional[str]:
        return self.timeline.dump() if self.timeline is not None else None

    def capture(self) -> None:
        self._captured = True
        e = self.engine
        # snapshot: warm-up steps must not change the model
        p0 = e.params.clone()
        r0 = e.running.clone()
        st0 = {k: v.clone() for k, v in self._opt_state().items()}
        s = torch.cuda.Stream(device=e.device)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(self._warmup_steps):
                self._launch()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        if self.use_graph:
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._launch()
            torch.cuda.synchronize()
        e.params.copy_(p0)
        e.running.copy_(r0)
        for k, v in self._opt_state().items():
            v.copy_(st0[k])
        e.sync_weights()
        torch.cuda.synchronize()

    def _opt_state(self):
        o = self.optimizer.opt if self._dist else self.optimizer
        return o.state

    def load(self, x_u8: torch.Tensor, labels: torch.Tensor) -> None:
        self.engine.set_input(x_u8, labels)

    def run(self) -> None:
        if not self._captured:
            self.capture()
        self.optimizer.begin_step()
        self.engine._step_count += 1
        if self.graph is not None:
            self.graph.replay()
        else:
            self._launch()
        self.steps += 1

    def result_async(self) -> torch.Tensor:
        """Enqueue the D2H copy of [sum loss, correct]; valid after the stream is synchronised."""
        self._host_stats.copy_(self.engine.stats, non_blocking=True)
        return self._host_stats

    def result(self) -> Tuple[float, float]:
        self.result_async()
        torch.cuda.current_stream().synchronize()
        b = self.engine.batch
        return float(self._host_stats[0]) / b, float(self._host_stats[1]) / b


class EngineEvalStep:
    """Inference / validation forward of a `ResNet50Engine` (BN folded to running statistics), CUDA-graphed."""

    def __init__(self, engine: ResNet50Engine, use_graph: bool = True):
        self.engine = engine
        self.use_graph = use_graph
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        engine.build(training=engine.grads is not None)
        self._host_stats = torch.zeros(2, dtype=torch.float32).pin_memory()

    def capture(self) -> None:
        e = self.engine
        s = torch.cuda.Stream(device=e.device)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            e.forward(training=False)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            e.forward(training=False)
        torch.cuda.synchronize()

    def run(self) -> None:
        if self.use_graph:
            if self.graph is None:
                self.capture()
            self.graph.replay()
        else:
            self.engine.forward(training=False)

    def result(self) -> Tuple[float, float]:
        self._host_stats.copy_(self.engine.stats, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        b = self.engine.batch
        return float(self._host_stats[0]) / b, float(self._host_stats[1]) / b
