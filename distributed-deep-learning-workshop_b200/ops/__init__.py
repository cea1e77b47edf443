"""Python entry points of the sm_100a kernels.

``ops.ext(name)`` loads (building in-tree if needed) one of the extensions:

    _b200_conv    tcgen05/TMEM/TMA implicit-GEMM convolution forward / dgrad / wgrad
    _b200_probe   hardware probes (UMMA descriptor addressing, TMA pipeline throughput); never on a hot path
    _b200_ops     BN / ReLU / pool / softmax-CE / preprocess kernels + fused optimizers
    _b200_comm    fused all-reduce kernels over NVLink symmetric memory
    _b200_loader  pinned-host ring buffer with side-stream H2D

On a box with a GPU the extensions are mandatory: a missing or unloadable binary raises instead of silently
falling back to eager PyTorch (``require_native``).
"""
from __future__ import annotations

from . import _build

EXT_NAMES = tuple(_build.EXTENSIONS)


def ext(name: str):
    return _build.load(name)


def build_all(verbose: bool = False) -> None:
    _build.build_all(verbose=verbose)


def native_available() -> bool:
    import torch

    return torch.cuda.is_available()


def require_native() -> None:
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("b200ddl: this code path needs a CUDA device (B200, sm_100a)")
    cap = torch.cuda.get_device_capability()
    if cap[0] != 10:
        raise RuntimeError(f"b200ddl: kernels are compiled for sm_100a only, found sm_{cap[0]}{cap[1]}")


def kernel_launches() -> int:
    """Total number of OUR kernels launched so far (what bench.py reports as gpu_launches)."""
    import sys

    n = 0
    for name in ("_b200_ops", "_b200_comm"):
        mod = sys.modules.get(name)
        if mod is not None:
            n += int(mod.launch_count())
    from . import conv as _conv

    n += _conv.plan_launches()
    return n
