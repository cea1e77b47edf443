"""Runner + distributed runtime on CPU (gloo, world_size 2) - the reference's HorovodRunner contract
(P1/03:391-417): closures travel by value, rank 0's return value comes back, any failing rank fails the gang."""
import os

import pytest

from b200ddl.parallel import Runner
from b200ddl.parallel.runner import RunnerError

BATCH_SIZE = 7  # driver-side global captured by the closure, like the notebook globals


def test_np_minus_one_runs_single_local_process():
    def fn():
        import b200ddl.parallel as hvd

        hvd.init()
        return hvd.rank(), hvd.size(), hvd.local_rank(), BATCH_SIZE

    assert Runner(np=-1, driver_log_verbosity="none", force_cpu=True).run(fn) == (0, 1, 0, 7)


def test_two_ranks_allreduce_broadcast_and_return_value():
    scale = 3.0

    def fn(offset):
        import torch
        import b200ddl.parallel as hvd

        hvd.init()
        t = torch.full((4,), float(hvd.rank() + offset))
        avg = hvd.allreduce(t, average=True)
        w = torch.full((3,), float(hvd.rank() + 5))
        hvd.broadcast(w, 0)
        objs = hvd.allgather_object({"rank": hvd.rank()})
        return {"avg": avg.tolist(), "w": w.tolist(), "size": hvd.size(), "objs": objs, "scale": scale}

    out = Runner(np=2, driver_log_verbosity="none", force_cpu=True).run(fn, offset=1.0)
    assert out["size"] == 2 and out["avg"] == [1.5] * 4 and out["w"] == [5.0] * 3
    assert [o["rank"] for o in out["objs"]] == [0, 1] and out["scale"] == 3.0


def test_gang_failure_surfaces_worker_traceback():
    def fn():
        import b200ddl.parallel as hvd

        hvd.init()
        if hvd.rank() == 1:
            raise ValueError("rank one exploded")
        import time

        time.sleep(30)
        return "never"

    r = Runner(np=2, driver_log_verbosity="none", force_cpu=True)
    with pytest.raises(RunnerError) as ei:
        r.run(fn)
    assert "rank one exploded" in str(ei.value) and "rank 1" in str(ei.value)


def test_distributed_optimizer_averages_gradients_and_keeps_replicas_identical():
    def fn():
        import torch
        import b200ddl.parallel as hvd
        from b200ddl import optim
        from b200ddl.train import Trainer
        from b200ddl.utils import checksum_across_ranks

        hvd.init()
        torch.manual_seed(100 + hvd.rank())  # different init per rank on purpose
        model = torch.nn.Sequential(torch.nn.Flatten(), torch.nn.Linear(3 * 8 * 8, 16), torch.nn.ReLU(),
                                    torch.nn.Linear(16, 4))
        opt = hvd.DistributedOptimizer(optim.SGD(0.1 * hvd.size(), momentum=0.9), bucket_mb=0.0001)
        tr = Trainer(model, device="cpu").compile(optimizer=opt)

        def ds():
            g = torch.Generator().manual_seed(hvd.rank())  # disjoint shards
            while True:
                y = torch.randint(0, 4, (8,), generator=g)
                x = (torch.randint(0, 30, (8, 8, 8, 3), generator=g) + (y * 50)[:, None, None, None]).to(torch.uint8)
                yield x, y

        h = tr.fit(ds(), steps_per_epoch=20, epochs=2, verbose=0,
                   callbacks=[hvd.callbacks.BroadcastGlobalVariablesCallback(0), hvd.callbacks.MetricAverageCallback()])
        same = checksum_across_ranks(tr.backend.flat.params)
        return {"same": same, "loss": h.history["loss"], "buckets": len(opt.buckets), "launches": opt.allreduce_launches}

    out = Runner(np=2, driver_log_verbosity="none", force_cpu=True).run(fn)
    assert out["same"], "replicas diverged"
    assert out["buckets"] >= 2 and out["launches"] >= 40 * out["buckets"] - 1
    assert out["loss"][-1] < out["loss"][0]


def test_learning_rate_warmup_ramps_from_lr_over_size_on_two_ranks():
    """`LearningRateWarmupCallback` (reference P1/03:315-318): with N ranks the LR starts at initial_lr / N, grows every
    batch, and is exactly initial_lr once the warm-up epochs are over - identically on every rank."""
    def fn():
        import torch
        import b200ddl.parallel as hvd
        from b200ddl import optim
        from b200ddl.train import LambdaCallback, Trainer

        hvd.init()
        torch.manual_seed(0)
        model = torch.nn.Sequential(torch.nn.Flatten(), torch.nn.Linear(3 * 8 * 8, 4))
        base_lr = 0.01 * hvd.size()
        opt = hvd.DistributedOptimizer(optim.SGD(base_lr))
        tr = Trainer(model, device="cpu").compile(optimizer=opt)
        seen = []
        rec = LambdaCallback(on_train_batch_end=lambda b, logs: seen.append(tr.optimizer.learning_rate))

        def ds():
            g = torch.Generator().manual_seed(hvd.rank())
            while True:
                y = torch.randint(0, 4, (8,), generator=g)
                yield torch.randint(0, 255, (8, 8, 8, 3), generator=g).to(torch.uint8), y

        tr.fit(ds(), steps_per_epoch=5, epochs=4, verbose=0,
               callbacks=[hvd.callbacks.BroadcastGlobalVariablesCallback(0),
                          hvd.callbacks.LearningRateWarmupCallback(initial_lr=base_lr, warmup_epochs=2), rec])
        lrs = torch.tensor(seen, dtype=torch.float64)
        gathered = [torch.zeros_like(lrs) for _ in range(hvd.size())]
        import torch.distributed as dist
        dist.all_gather(gathered, lrs)
        return {"lrs": seen, "base": base_lr, "size": hvd.size(), "same": all(torch.equal(gathered[0], t) for t in gathered)}

    out = Runner(np=2, driver_log_verbosity="none", force_cpu=True).run(fn)
    lrs, base = out["lrs"], out["base"]
    assert out["size"] == 2 and out["same"] and len(lrs) == 20
    assert abs(lrs[0] - base / 2) < 1e-12                       # first batch: initial_lr / size
    warm = lrs[:10]
    assert all(b > a for a, b in zip(warm, warm[1:]))           # strictly increasing during the 2 warm-up epochs
    assert warm[-1] < base
    assert all(abs(v - base) < 1e-12 for v in lrs[10:])         # exactly initial_lr afterwards


def test_hung_rank_hits_the_timeout_and_no_worker_survives(tmp_path):
    """Failure detection (SURVEY.md 5.3): a rank that hangs (not crashes) is caught by `timeout_s`; the error says so and
    every worker process the Runner started is gone afterwards."""
    import os
    import time

    piddir = str(tmp_path)

    def fn():
        import os
        import time
        import b200ddl.parallel as hvd

        hvd.init()
        with open(os.path.join(piddir, f"pid_{hvd.rank()}"), "w") as f:
            f.write(str(os.getpid()))
        if hvd.rank() == 1:
            time.sleep(3600)          # the hang: rank 0 waits for it in the barrier below
        hvd.barrier()
        return "unreachable"

    t0 = time.time()
    with pytest.raises(RunnerError) as ei:
        Runner(np=2, driver_log_verbosity="none", force_cpu=True, timeout_s=20).run(fn)
    assert "timed out after 20" in str(ei.value)
    assert time.time() - t0 < 90
    pids = [int(open(os.path.join(piddir, f"pid_{r}")).read()) for r in (0, 1)]
    deadline = time.time() + 10
    alive = pids
    while alive and time.time() < deadline:
        alive = []
        for pid in pids:
            try:
                os.kill(pid, 0)       # signal 0: existence check only
                alive.append(pid)
            except ProcessLookupError:
                pass
        time.sleep(0.2)
    assert not alive, f"worker processes still alive after the timeout: {alive}"


def test_workers_get_their_share_of_the_cores(monkeypatch):
    """Each rank's OpenMP team is sized cores // ranks unless OMP_NUM_THREADS was set by the user (torchrun does the same;
    full-size teams in every rank oversubscribe the host)."""
    import os

    def fn():
        import os
        import torch
        import b200ddl.parallel as hvd

        hvd.init()
        return os.environ.get("OMP_NUM_THREADS"), torch.get_num_threads()

    from b200ddl.utils.cpus import usable_cpus

    monkeypatch.delenv("OMP_NUM_THREADS", raising=False)
    monkeypatch.delenv("MKL_NUM_THREADS", raising=False)   # torch sizes its team from MKL_NUM_THREADS when that is set
    share = max(1, usable_cpus() // 2)
    env_val, torch_threads = Runner(np=2, driver_log_verbosity="none", force_cpu=True).run(fn)
    assert env_val == str(share) and torch_threads == share
    monkeypatch.setenv("OMP_NUM_THREADS", "3")           # an explicit user setting wins
    assert Runner(np=2, driver_log_verbosity="none", force_cpu=True).run(fn)[0] == "3"


def test_persistent_rank_pool_reuses_processes_and_process_group():
    """`Runner(persistent=True)`: the same rank processes (and their process group) serve several `run()` calls - what
    back-to-back HPO trials over the distributed trainer use; a failing job stops the gang and the next call gets a new one."""
    import time

    def fn(offset):
        import os

        import torch
        import b200ddl.parallel as hvd

        hvd.init()
        s = hvd.allreduce(torch.ones(2) * (hvd.rank() + offset), average=False)
        return os.getpid(), float(s[0])

    with Runner(np=2, driver_log_verbosity="none", force_cpu=True, persistent=True) as r:
        pid0, v0 = r.run(fn, offset=1.0)
        assert v0 == 3.0 and r.last_timing["pool_started"] is True
        t0 = time.time()
        pid1, v1 = r.run(fn, offset=2.0)
        dt = time.time() - t0
        assert pid1 == pid0 and v1 == 5.0 and r.last_timing["pool_started"] is False
        assert dt < r.last_timing["pool_start_s"] + 2.0  # no spawn / import / rendezvous the second time

        def bad():
            import b200ddl.parallel as hvd

            hvd.init()
            if hvd.rank() == 1:
                raise ValueError("second job exploded")
            import time as _t

            _t.sleep(30)

        with pytest.raises(RunnerError) as ei:
            r.run(bad)
        assert "second job exploded" in str(ei.value)
        pid2, v2 = r.run(fn, offset=1.0)   # a fresh gang
        assert pid2 != pid0 and v2 == 3.0


def test_consolidate_state_completes_rank_sharded_momentum_and_save_refuses_a_sharded_state(tmp_path):
    """`fused_update` shards the momentum over ranks (csrc/allreduce.cu allreduce_sgd_nvls_kernel updates only the owner's
    slice).  `consolidate_state()` must rebuild the complete tensor on every rank from the owners' slices, `Trainer.save`
    must refuse an unconsolidated state, and `broadcast_parameters` must consolidate first.  The kernel needs NVLS; the
    slice logic is exercised here on 2 CPU ranks by putting the optimizer into the sharded state by hand."""
    ck = str(tmp_path / "ck.pt")

    def fn(ck):
        import torch
        import b200ddl.parallel as hvd
        from b200ddl import optim
        from b200ddl.train import Trainer

        hvd.init()
        torch.manual_seed(0)
        model = torch.nn.Sequential(torch.nn.Flatten(), torch.nn.Linear(3 * 8 * 8, 16), torch.nn.ReLU(), torch.nn.Linear(16, 4))
        opt = hvd.DistributedOptimizer(optim.SGD(0.1, momentum=0.9), bucket_mb=0.0001)
        tr = Trainer(model, device="cpu").compile(optimizer=opt)
        x = torch.randint(0, 255, (8, 8, 8, 3), dtype=torch.uint8)
        y = torch.randint(0, 4, (8,))
        tr.fit([(x, y)] * 2, steps_per_epoch=2, epochs=1, verbose=0)      # buckets exist, momentum is allocated
        mom = opt.opt.state["momentum"]
        truth = torch.arange(mom.numel(), dtype=torch.float32) * 0.5 + 1.0
        # emulate the sharded state: a rank holds the truth on the ranges it owns and garbage everywhere else
        opt.fused_update = True
        opt._state_complete = False
        mom.fill_(-777.0 - hvd.rank())
        covered = torch.zeros(mom.numel(), dtype=torch.bool)
        for b in opt.buckets:
            a, e = opt.owned_range(b.lo, b.hi, hvd.rank(), hvd.size())
            mom[a:e] = truth[a:e]
            for r in range(hvd.size()):
                a2, e2 = opt.owned_range(b.lo, b.hi, r, hvd.size())
                covered[a2:e2] = True
        refused = False
        try:
            tr.save(ck + f".{hvd.rank()}")
        except RuntimeError as ex:
            refused = "consolidate_state" in str(ex)
        opt.consolidate_state()
        ok = bool(torch.equal(mom[covered], truth[covered])) and not opt.state_is_sharded
        tr.save(ck + f".{hvd.rank()}")                                     # complete state: accepted
        # a later fused step shards it again; broadcast_parameters consolidates before it broadcasts
        opt.begin_step()
        sharded_again = opt.state_is_sharded
        mom.fill_(-1.0)
        for b in opt.buckets:
            a, e = opt.owned_range(b.lo, b.hi, hvd.rank(), hvd.size())
            mom[a:e] = truth[a:e] * 2
        opt.broadcast_parameters(tr.backend.flat.params, 0)
        ok2 = bool(torch.equal(mom[covered], truth[covered] * 2))
        return {"refused": refused, "ok": ok, "sharded_again": sharded_again, "ok2": ok2, "n": int(covered.sum()), "buckets": len(opt.buckets)}

    out = Runner(np=2, driver_log_verbosity="none", force_cpu=True).run(fn, ck=ck)
    assert out["refused"] and out["ok"] and out["sharded_again"] and out["ok2"], out
    assert out["buckets"] >= 2 and out["n"] > 0
