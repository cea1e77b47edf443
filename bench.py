#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): ResNet-50 training images/sec, bf16, 224x224 synthetic images, per-GPU batch
256 (reference P1/03:81), N = 1/2/4/8 B200 (weak scaling), device-timed, max over ranks.

    python bench.py [--gpus N --steps K --warmup W]            # our engine (N>1: launched by torchrun)
    python bench.py --impl reference ...                        # the unmodified reference (not installable offline)
    python bench.py --impl torch-baseline ...                   # operative baseline: torch + cuDNN + NCCL (BASELINE.md §2)

Prints ONE JSON line on rank 0.  `value` = kernel-only device time of K full training steps (forward, backward,
fused all-reduce, optimizer) with the step captured in a CUDA graph and the input batch resident on the device;
`e2e` = the same metric through the public API (`Trainer.fit` over the pinned ring loader): every step includes the
host->device copy of its input batch from pinned memory and a device->host read of the step's loss/accuracy.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "resnet50_train_images_per_sec"


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int = 0):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for nme, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm_sorted = sorted(sm)
        # median over samples taken under load (power above idle)
        loaded = [s for s, p in zip(sm, power) if p > 300.0] or sm
        loaded.sort()
        return {"sm_mhz": loaded[len(loaded) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power), "sm_mhz_min": sm_sorted[0]}


def run_reference(args):
    # The reference tree holds Databricks notebooks only: no setup.py / pyproject, and its imports (tensorflow,
    # horovod, petastorm, pyspark, mlflow, hyperopt) are absent from the image and the offline wheelhouse.
    if int(os.environ.get("RANK", "0")) != 0:   # launched under torchrun for N > 1 like our own arm: ONE line, from rank 0
        return 0
    print(json.dumps({"impl": "reference", "unavailable": "reference is 11 Databricks notebooks with no installable "
                      "package (pip: neither setup.py nor pyproject.toml); TensorFlow/Horovod/Spark/Petastorm/MLflow "
                      "are not in the image or /opt/wheelhouse (see DESIGN.md)"}))
    return 0


def run_baseline_child(args, rank: int, world: int):
    """Operative baseline in THE SAME invocation (same box, same lease, same N / steps / warm-up): every rank spawns
    `baseline/torch_resnet50.py` as its own child process (fresh CUDA context + NCCL group on MASTER_PORT + 23) once our
    arm has finished; the child samples its own clocks during its timed region.  Returns rank 0's parsed JSON line.
    First attempt captures the step in a CUDA graph; if that child fails, one retry without the graph."""
    script = os.path.join(ROOT, "baseline", "torch_resnet50.py")
    # torchrun's variables must not leak into the children: with TORCHELASTIC_USE_AGENT_STORE=True, init_process_group
    # would look for the AGENT's TCPStore on our new port (nobody serves one there) and wait for its timeout
    env = {k: v for k, v in os.environ.items() if not k.startswith(("TORCHELASTIC_", "TORCH_NCCL_ASYNC", "GROUP_", "ROLE_"))}
    env["RANK"], env["WORLD_SIZE"] = str(rank), str(world)
    env["LOCAL_WORLD_SIZE"] = str(world)
    env["LOCAL_RANK"] = os.environ.get("LOCAL_RANK", str(rank))
    env.setdefault("MASTER_ADDR", "127.0.0.1")
    base_port = int(os.environ.get("MASTER_PORT", "29500"))
    result, notes = None, []
    # N = 1: CUDA graph first, eager as the fallback.  N > 1: eager only - capturing the hook-launched NCCL all-reduces of
    # the baseline in a CUDA graph did not complete on the 4-GPU box (child timed out at 150 s, profiles/r2_bench_w4.json);
    # eager costs the baseline ~4 % at N = 1 (4,710 vs 4,891 img/s in round 1), it is what DDP users run.
    for attempt, graph in enumerate((True, False) if world == 1 else (False,)):
        env["MASTER_PORT"] = str(base_port + 23 + attempt)
        cmd = [sys.executable, script, "--steps", str(args.steps), "--warmup", str(args.warmup), "--batch",
               str(args.batch), "--classes", str(args.classes)] + (["--graph"] if graph else [])
        timed_out = False
        try:
            p = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=args.baseline_timeout)
            rc, out, err = p.returncode, p.stdout, p.stderr
        except subprocess.TimeoutExpired as ex:
            rc, out, err, timed_out = -9, (ex.stdout or ""), "timeout", True
            if isinstance(out, bytes):
                out = out.decode(errors="replace")
        ok_all = _all_ranks_ok(rc == 0, world)
        if rank == 0 and rc == 0:
            for ln in out.splitlines():
                if ln.startswith("{"):
                    result = json.loads(ln)
        if ok_all and (rank != 0 or result is not None):
            break
        notes.append(f"attempt graph={graph} failed rc={rc}: {str(err)[-300:]}")
        result = None
        if not _all_ranks_ok(not timed_out, world):
            break  # a hang would most likely repeat: never spend a second timeout (the driver's own limit is close)
    if rank == 0 and result is not None and notes:
        result["notes"] = notes
    if rank == 0 and result is None:
        result = {"unavailable": "; ".join(notes)[-600:]}
    return result


def _all_ranks_ok(ok: bool, world: int) -> bool:
    """Agreement between the rank processes WITHOUT a live process group (ours is already shut down): files in /tmp."""
    if world == 1:
        return ok
    import tempfile

    # all ranks of one launch share the torchrun agent as parent: unique per launch, equal across ranks
    tag = os.environ.get("MASTER_PORT", "0") + "_" + str(os.getppid())
    d = os.path.join(tempfile.gettempdir(), f"b200ddl_bench_{tag}")
    os.makedirs(d, exist_ok=True)
    rk = os.environ.get("RANK", "0")
    seq = getattr(_all_ranks_ok, "seq", 0)
    _all_ranks_ok.seq = seq + 1
    with open(os.path.join(d, f"{seq}_{rk}"), "w") as f:
        f.write("1" if ok else "0")
    t0 = time.time()
    while time.time() - t0 < 120:
        have = [os.path.join(d, f"{seq}_{r}") for r in range(world)]
        if all(os.path.exists(h) and os.path.getsize(h) > 0 for h in have):
            return all(open(h).read().strip() == "1" for h in have)
        time.sleep(0.2)
    return False


def run_torch_baseline(args):
    sys.argv = [sys.argv[0], "--steps", str(args.steps), "--warmup", str(args.warmup), "--batch", str(args.batch),
                "--classes", str(args.classes)] + (["--graph"] if args.graph_baseline else [])
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import torch_resnet50

    torch_resnet50.main(sys.argv[1:])
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=256, help="per-GPU batch (reference P1/03:81)")
    ap.add_argument("--classes", type=int, default=1000)
    ap.add_argument("--impl", default="b200ddl", choices=["b200ddl", "reference", "torch-baseline"])
    ap.add_argument("--algo", default="auto", help="all-reduce: auto|nvls|p2p|oneshot|nccl")
    ap.add_argument("--bucket-mb", type=float, default=16.0)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--graph-baseline", action="store_true")
    ap.add_argument("--optimizer", default="sgd", choices=["sgd", "adam"])
    ap.add_argument("--no-fuse-bwd-reduce", action="store_true")
    ap.add_argument("--fuse-bn-coeffs", action="store_true", help="opt-in: BN coefficients inside the apply kernels (measured slower)")
    ap.add_argument("--overlap-wgrad", action="store_true", help="(default; kept for old command lines) weight-gradient GEMMs on a side stream")
    ap.add_argument("--no-overlap-wgrad", action="store_true", help="issue the weight-gradient GEMMs in line on the compute stream")
    ap.add_argument("--wgrad-smem", type=int, default=0)
    ap.add_argument("--fused-update", action="store_true", help="all-reduce + SGD + weight multicast in one kernel")
    ap.add_argument("--no-baseline", action="store_true", help="skip the same-lease torch+cuDNN+NCCL baseline child")
    ap.add_argument("--baseline-timeout", type=int, default=200)
    ap.add_argument("--no-block-grad", action="store_true", help="A/B: block-gradient merge as separate reduce passes")
    ap.add_argument("--stem-bwd-fuse", action="store_true", help="A/B (opt-in): max-pool backward fused with the stem-BN backward")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step computed as "
                                                         "DIR/<name>.npy (rank 0), to compare two builds output for output")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "torch-baseline":
        return run_torch_baseline(args)

    import torch

    import b200ddl
    from b200ddl import ops, optim
    from b200ddl import parallel as dist
    from b200ddl.loader import SyntheticDataset
    from b200ddl.models.resnet_engine import ResNet50Engine
    from b200ddl.train import Trainer

    dist.init()
    rank, world = dist.rank(), dist.size()
    if world != args.gpus and rank == 0 and "WORLD_SIZE" in os.environ:
        print(f"# note: --gpus {args.gpus} but WORLD_SIZE={world}", file=sys.stderr)
    dev = dist.device()
    torch.backends.cudnn.benchmark = True

    engine = ResNet50Engine(batch=args.batch, num_classes=args.classes, device=dev, seed=0, max_ctas=0,
                            overlap_wgrad=not args.no_overlap_wgrad, wgrad_smem_budget=args.wgrad_smem,
                            fuse_bwd_reduce=not args.no_fuse_bwd_reduce, fuse_bn_coeffs=args.fuse_bn_coeffs,
                            fuse_block_grad=False if args.no_block_grad else None,
                            fuse_stem_bwd=True if args.stem_bwd_fuse else None)
    lr = 0.1 * world  # LR x world size (reference P1/03:301)
    base_opt = optim.SGD(lr, momentum=0.9, weight_decay=1e-4) if args.optimizer == "sgd" else optim.Adam(1e-3 * world)
    opt = (dist.DistributedOptimizer(base_opt, bucket_mb=args.bucket_mb, algo=args.algo, fused_update=args.fused_update)
           if world > 1 else base_opt)
    trainer = Trainer(engine, use_graph=not args.no_graph)
    trainer.compile(optimizer=opt, loss="sparse_categorical_crossentropy", metrics=["accuracy"])
    if world > 1:
        trainer.broadcast_state(0)
    step = trainer.backend.step

    # ---------------------------------------------------------------- kernel-only timed region
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    x = torch.randint(0, 256, (args.batch, 224, 224, 3), device=dev, dtype=torch.uint8, generator=g)
    y = torch.randint(0, args.classes, (args.batch,), device=dev, generator=g)
    step.load(x, y)
    n0 = ops.kernel_launches()
    step.capture()
    launches_per_step = (ops.kernel_launches() - n0) // (step._warmup_steps + (1 if step.graph is not None else 0))
    for _ in range(args.warmup):
        step.run()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(torch.cuda.current_device())
    if rank == 0:
        sampler.start()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step.run()
    e1.record()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    ms = float(dist.allreduce(ms, average=False).item()) if world == 1 else float(_max_over_ranks(ms))
    loss, acc = step.result()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, engine, loss, acc)
    # outside the timed region: after K data-parallel steps every rank must hold bit-identical fp32 master weights
    # (a gradient that was all-reduced before its producer finished would show up here)
    from b200ddl.utils import checksum_across_ranks
    params_identical = bool(checksum_across_ranks(engine.params)) if world > 1 else None
    global_batch = args.batch * world
    value = global_batch * args.steps / (ms / 1e3)

    # ---------------------------------------------------------------- end-to-end through the public API
    e2e = None
    if not args.no_e2e:
        ds = SyntheticDataset(args.batch, num_classes=args.classes, device=dev, cur_shard=rank, shard_count=world,
                              threads=6, pool_images=4096, seed=7)
        with ds:
            trainer.fit(ds, steps_per_epoch=args.warmup, epochs=1, verbose=0)  # warm the loader + host path
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            b0 = ds.ring.h2d_bytes
            t0 = time.perf_counter()
            f0 = torch.cuda.Event(enable_timing=True)
            f1 = torch.cuda.Event(enable_timing=True)
            f0.record()
            hist = trainer.fit(ds, steps_per_epoch=args.steps, epochs=1, verbose=0)
            f1.record()
            torch.cuda.synchronize()
            wall_ms = (time.perf_counter() - t0) * 1e3
            ems = max(f0.elapsed_time(f1), wall_ms)
            ems = float(_max_over_ranks(torch.tensor([ems], device=dev))) if world > 1 else ems
            h2d = (ds.ring.h2d_bytes - b0) // args.steps
            e2e = {"value": global_batch * args.steps / (ems / 1e3), "unit": "images/s",
                   "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 8, "ms_per_step": ems / args.steps,
                   "api": "b200ddl.train.Trainer.fit over loader.SyntheticDataset (pinned ring, side-stream H2D)",
                   "loader_wait_ms": ds.ring.consumer_wait_ms, "final_loss": hist.history["loss"][-1]}

    cfg_flags = {"fuse_block_grad": bool(engine.fuse_block_grad), "fuse_stem_bwd": bool(engine.fuse_stem_bwd),
                 "bn_rows_unroll": int(engine._e.get_bn_rows_unroll()) if hasattr(engine._e, "get_bn_rows_unroll") else 1}
    # ---------------------------------------------------------------- same-lease baseline (torch + cuDNN + NCCL)
    baseline = None
    algo_used = getattr(opt, "algo", "none") if world > 1 else "none"
    fused_used = bool(getattr(opt, "fused_update", False))
    # release the CUDA graph (it may hold captured NCCL work with --algo nccl), the engine and the symmetric buffers BEFORE
    # the process group goes away, then the group itself
    del trainer, step, engine, opt, base_opt
    import gc

    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    dist.shutdown()
    if not args.no_baseline:
        baseline = run_baseline_child(args, rank, world)
    if rank == 0:
        vs = None
        if baseline is not None and baseline.get("value"):
            vs = value / float(baseline["value"])
        out = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": vs,
            "baseline": (None if baseline is None else {
                "what": "torchvision ResNet-50, bf16 autocast, channels_last, cuDNN, fused SGD, flat-gradient views, "
                        "NCCL all_reduce per bucket + div overlapped from grad hooks (Horovod path, reference P1/03:301-302), "
                        "CUDA graph when capturable; run as a child process in this same invocation",
                **{k: baseline.get(k) for k in ("value", "ms_per_step", "clocks", "graph", "n_gpus", "steps", "warmup",
                                                "config", "notes", "unavailable") if k in baseline}}),
            "dtype": "bf16", "data": "synthetic uint8 224x224x3 images, random-init weights",
            "impl": "b200ddl",
            "config": {"model": "resnet50", "global_batch": global_batch, "per_gpu_batch": args.batch,
                       "image": "224x224x3", "classes": args.classes, "parallelism": f"dp{world}",
                       "optimizer": args.optimizer, "allreduce": algo_used,
                       "fused_allreduce_sgd": fused_used,
                       "cuda_graph": not args.no_graph, "overlap_wgrad": not args.no_overlap_wgrad, **cfg_flags,
                       "l2": "activations per step are several GB (>> 126 MB L2); no explicit flush needed"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches_per_step * args.steps),
            "launches_per_step": int(launches_per_step), "loss": loss, "accuracy": acc,
            "params_identical_across_ranks": params_identical,
        }
        print(json.dumps(out), flush=True)
    dist.shutdown()
    return 0


DUMP_WEIGHT_SAMPLE = 1 << 22   # 16 MB of the 25.6 M fp32 weights (102 MB): the dump stays far below 64 MB


def dump_outputs(out_dir: str, engine, loss: float, acc: float) -> None:
    """Write what a training step hands its caller, as it stands after the last timed step: loss and accuracy, the fp32
    logits, the BatchNorm running statistics and a fixed, seeded sample of the updated fp32 weights.  Tensors are taken
    in torchvision names and layouts and concatenated in name order, so two builds compare element for element even
    when their internal parameter layouts differ.  Compare with a tolerance: the reductions use floating-point atomics,
    so two runs of one build already differ after a few dozen training steps."""
    import numpy as np
    import torch

    sd = engine.state_dict()
    stats = sorted(k for k in sd if k.endswith((".running_mean", ".running_var")))
    weights = sorted(set(sd) - set(stats))
    w = torch.cat([sd[k].reshape(-1) for k in weights]).numpy()
    idx = np.sort(np.random.default_rng(0).choice(w.size, min(DUMP_WEIGHT_SAMPLE, w.size), replace=False))
    arrays = {"loss": np.array([loss], np.float64), "accuracy": np.array([acc], np.float64),
              "logits": engine.logits.float().cpu().numpy(),
              "bn_running_stats": torch.cat([sd[k].reshape(-1) for k in stats]).numpy(),
              "weights_sample": w[idx]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _max_over_ranks(t):
    import torch.distributed as td

    td.all_reduce(t, op=td.ReduceOp.MAX)
    return t.item()


if __name__ == "__main__":
    sys.exit(main())
