"""GPU tests (run on the B200 box: `pytest tests -m gpu`): every hand-written kernel against a PyTorch fp32
reference of the same op, plus the ResNet-50 engine against torchvision with identical weights."""
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))


@pytest.fixture(scope="module")
def checks():
    import gpu_check

    return gpu_check


def test_native_extensions_are_loaded():
    from b200ddl import ops

    ops.require_native()
    for n in ops.EXT_NAMES:
        m = ops.ext(n)
        assert m.__file__.endswith(".so") and "csrc/build" in m.__file__


def test_elementwise_and_optimizer_kernels(checks):
    assert checks.case_elementwise()


def test_conv_forward_tcgen05(checks):
    assert checks.case_conv_fwd()


def test_conv_dgrad_tcgen05(checks):
    assert checks.case_conv_dgrad()


def test_conv_2d_halo_opt_in(checks, monkeypatch):
    """Opt-in path (B200DDL_HALO2D=1): (8, bh, 1) boxes, one [10 x (bh+2)] halo load per tile, strided row-shifted UMMA
    descriptors - forward, statistics, dgrad and the fused dgrad reduction against the fp32 references."""
    monkeypatch.setenv("B200DDL_HALO2D", "1")
    assert checks.case_conv_fwd()
    assert checks.case_conv_dgrad()


def test_conv_wgrad_tcgen05(checks):
    assert checks.case_conv_wgrad()


def test_stem_conv_tcgen05(checks):
    assert checks.case_stem()


def test_block_gradient_epilogue(checks):
    """conv1 dgrad with the fused block-gradient merge (skip add + ReLU bitmask + bn3 reduction), dense and compact skip,
    partial last tile, and the benchmark shape at batch 256."""
    assert checks.case_block_grad()


def test_classifier_head_on_tcgen05(checks):
    """FC forward / dgrad / wgrad on the implicit-GEMM kernels + softmax_ce_head + fc_bias_grad vs torch fp32."""
    assert checks.case_head()


def test_inference_epilogue_and_fused_inference_engine(checks):
    """conv epilogue with folded BatchNorm + activation (+ residual) vs fp32; inference-built engine vs eval on the training build."""
    assert checks.case_fused_infer()


def test_reference_model_mobilenetv2_on_native_kernels(checks):
    """Frozen MobileNetV2 base + Dense head: depthwise / stem kernels and the whole engine vs the torch.nn module."""
    assert checks.case_mobilenet()


def test_conv_numerics_at_benchmark_batch(checks):
    """forward (+statistics) / dgrad / wgrad vs fp32 at the batch-256 layer shapes the benchmark runs."""
    assert checks.case_big_numerics()


def test_resnet50_engine_unfused_block_gradient_matches_torchvision(checks):
    """A/B path: block-gradient merge as separate reduce passes (fuse_block_grad=False)."""
    assert checks.case_engine(quick=True, fuse_block_grad=False)


def test_resnet50_engine_matches_torchvision(checks):
    assert checks.case_engine()


def test_resnet50_engine_inline_wgrad_matches_torchvision(checks):
    """Same gradient criteria with the weight-gradient GEMMs issued in line instead of on the side stream."""
    assert checks.case_engine(overlap_wgrad=False, quick=True)


def test_ring_loader_h2d_roundtrip():
    from b200ddl.loader import SyntheticDataset

    with SyntheticDataset(batch_size=16, num_classes=10, image_size=(64, 64), threads=2, pool_images=64) as ds:
        seen = []
        for _ in range(6):
            x, y = next(ds)
            assert x.is_cuda and x.shape == (16, 64, 64, 3) and x.dtype == torch.uint8
            assert y.is_cuda and int(y.min()) >= 0 and int(y.max()) < 10
            seen.append(int(x.sum()))
        assert ds.ring.h2d_bytes == 6 * 16 * (64 * 64 * 3 + 8)
    assert len(set(seen)) > 1


def test_gpu_jpeg_decode_dataset_matches_cpu_decode(tmp_path):
    """`make_dataset(decode='gpu')`: nvJPEG decode + our planar->HWC bilinear resize kernel vs the CPU (PIL) pipeline -
    same rows, same labels, pixels equal up to decoder / resampler rounding."""
    from b200ddl import Session
    from b200ddl.data import col, pandas_udf, synthetic_images
    from b200ddl.loader import make_converter

    Session(user="gpu@example.com", root=str(tmp_path))
    raw = synthetic_images(64, size=(96, 80), jpeg=True, seed=4)   # stored 96x80, served at 64x64: the resize kernel runs

    @pandas_udf("int")
    def label_idx(path):
        return path.map(lambda p: hash(p.split("/")[-2]) % 5)

    t = raw.withColumn("label_idx", label_idx(col("path"))).select(["content", "label_idx"])
    conv = make_converter(t, str(tmp_path / "cache"))
    with conv.make_dataset(batch_size=16, num_epochs=1, workers_count=1, image_size=(64, 64)) as cpu_ds, \
         conv.make_dataset(batch_size=16, num_epochs=1, image_size=(64, 64), decode="gpu") as gpu_ds:
        n = 0
        for (xc, yc), (xg, yg) in zip(cpu_ds, gpu_ds):
            assert xg.is_cuda and xg.dtype == torch.uint8 and xg.shape == (16, 64, 64, 3)
            assert torch.equal(yc.cpu(), yg.cpu())
            diff = (xc.cpu().float() - xg.cpu().float()).abs()
            assert diff.mean() < 3.0 and diff.max() < 48.0, (float(diff.mean()), float(diff.max()))
            n += 1
        assert n == 4 and gpu_ds.gpu_decoded == 64 and gpu_ds.cpu_decoded == 0 and gpu_ds.compressed_bytes > 0
        print("GPU JPEG backend:", gpu_ds.backend, gpu_ds.backend_errors)
        assert gpu_ds.backend.startswith("nvjpeg:"), (gpu_ds.backend, gpu_ds.backend_errors)   # the native decoder, not the fallback
    conv.delete()


def test_batched_resize_kernel_matches_pil_bilinear():
    """csrc/jpeg_resize.cu: one launch resizes images of DIFFERENT sizes; the filter is PIL's BILINEAR (support stretched by
    the down-scale factor), so it must agree with `Image.resize(..., BILINEAR)` to within rounding for shrink and enlarge."""
    import numpy as np
    from PIL import Image

    from b200ddl import ops

    jpeg = ops.ext("_b200_jpeg")
    rng = np.random.default_rng(0)
    sizes = [(375, 500), (96, 80), (224, 224), (100, 300), (600, 800), (50, 60)]
    imgs, table, off = [], [], 0
    for h, w in sizes:
        base = rng.integers(0, 255, (h // 8 + 1, w // 8 + 1, 3)).astype(np.uint8)
        img = np.asarray(Image.fromarray(base).resize((w, h), Image.BICUBIC)).astype(np.int32)
        img = np.clip(img + rng.integers(-20, 20, img.shape), 0, 255).astype(np.uint8)
        imgs.append(img)
        table += [off, w, h, w * 3]
        off += (h * w * 3 + 255) // 256 * 256
    src = torch.zeros(off, dtype=torch.uint8)
    for img, o in zip(imgs, table[0::4]):
        src[o:o + img.size] = torch.from_numpy(img.reshape(-1))
    out = torch.empty(len(sizes), 224, 224, 3, device="cuda", dtype=torch.uint8)
    jpeg.resize_batched(src.cuda(), torch.tensor(table, dtype=torch.int64, device="cuda"), out)
    for i, img in enumerate(imgs):
        ref = np.asarray(Image.fromarray(img).resize((224, 224), Image.BILINEAR)).astype(np.int32)
        d = np.abs(out[i].cpu().numpy().astype(np.int32) - ref)
        assert d.max() <= 2 and d.mean() < 0.4, (sizes[i], int(d.max()), float(d.mean()))


def test_smoke_entry():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g

    g.smoke()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_fused_allreduce_two_gpus():
    import subprocess

    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29611",
                        os.path.join(ROOT, "benchmarks", "allreduce_check.py"), "--quick"],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]
    assert "ALLREDUCE CHECK PASS" in p.stdout


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_fused_allreduce_sgd_matches_unfused_two_gpus():
    """all-reduce + SGD-momentum + weight multicast in ONE kernel == NCCL average followed by a plain fp32 update."""
    import subprocess

    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29733",
                        os.path.join(ROOT, "benchmarks", "fused_update_check.py")],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "FUSED UPDATE CHECK PASS" in p.stdout or "UNAVAILABLE" in p.stdout


def _torchrun(nproc: int, script: str, *args: str, port: int = 29800, timeout: int = 900):
    import subprocess

    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
                           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, script), *args],
                          capture_output=True, text=True, timeout=timeout, cwd=ROOT)


@pytest.mark.parametrize("world", [4, 8])
def test_fused_allreduce_broadcast_and_replicas_multi_gpu(world):
    """4- and 8-GPU boxes: every comm kernel (one-shot / two-shot P2P / NVLS, symmetric broadcast, DistributedOptimizer on each
    algorithm) against NCCL, bit-identical across ranks; then a short data-parallel training run whose fp32 master
    weights must be bit-identical on all ranks."""
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    p = _torchrun(world, "benchmarks/allreduce_check.py", "--quick", "--max-mb", "64", port=29811 + world)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]
    assert "ALLREDUCE CHECK PASS" in p.stdout
    p = _torchrun(world, "bench.py", "--gpus", str(world), "--steps", "4", "--warmup", "3", "--no-e2e", "--no-baseline",
                  port=29851 + world)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]
    import json

    line = [l for l in p.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["n_gpus"] == world and d["params_identical_across_ranks"] is True and d["loss"] == d["loss"]
