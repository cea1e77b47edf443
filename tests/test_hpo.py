"""HPO (reference Hyperopt usage: P2/01:194-243, P2/02:322-370)."""
import math
import threading
import time

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from b200ddl import hpo, tracking
from b200ddl.hpo import STATUS_FAIL, STATUS_OK, ParallelTrials, Trials, fmin, hp, rand, space_eval, tpe

SPACE = {"optimizer": hp.choice("optimizer", ["Adadelta", "Adam"]),
         "learning_rate": hp.loguniform("learning_rate", -5, 0),
         "dropout": hp.uniform("dropout", 0.1, 0.9)}


def test_samplers_respect_bounds():
    rng = np.random.default_rng(0)
    nodes = hpo._nodes(SPACE)
    for _ in range(200):
        v = rand.suggest(nodes, Trials(), rng)
        assert v["optimizer"] in (0, 1)
        assert math.exp(-5) <= v["learning_rate"] <= 1.0
        assert 0.1 <= v["dropout"] <= 0.9


@settings(max_examples=25, deadline=None)
@given(low=st.floats(-10, 0), span=st.floats(0.1, 5), q=st.sampled_from([0.5, 1.0, 8.0]))
def test_quniform_is_quantised(low, span, q):
    n = hp.quniform("x", low, low + span, q)
    v = hpo._sample_node(n, np.random.default_rng(1))
    assert abs(v / q - round(v / q)) < 1e-9


def test_fmin_returns_choice_index_and_space_eval():
    def obj(p):
        return {"loss": (p["dropout"] - 0.3) ** 2 + (0 if p["optimizer"] == "Adam" else 1), "status": STATUS_OK}

    trials = Trials()
    best = fmin(obj, SPACE, algo=tpe.suggest, max_evals=60, trials=trials, rstate=0)
    assert best["optimizer"] == 1                        # index, not 'Adam' (Hyperopt behaviour, Q7)
    assert space_eval(SPACE, best)["optimizer"] == "Adam"
    assert abs(best["dropout"] - 0.3) < 0.15
    assert len(trials) == 60 and trials.best_trial["result"]["loss"] < 0.03


def test_tpe_beats_random_on_quadratic():
    space = {"x": hp.uniform("x", -10, 10), "y": hp.uniform("y", -10, 10)}
    f = lambda p: (p["x"] - 3) ** 2 + (p["y"] + 2) ** 2
    res = {"tpe": [], "rand": []}
    for seed in range(5):
        for name, algo in (("tpe", tpe), ("rand", rand)):
            t = Trials()
            fmin(f, space, algo=algo.suggest, max_evals=80, trials=t, rstate=seed)
            res[name].append(t.best_trial["result"]["loss"])
    assert np.median(res["tpe"]) < np.median(res["rand"])


def test_failed_trials_are_recorded_not_fatal():
    def obj(p):
        if p["x"] > 0.5:
            raise RuntimeError("boom")
        return p["x"]

    t = Trials()
    best = fmin(obj, {"x": hp.uniform("x", 0, 1)}, algo=rand.suggest, max_evals=30, trials=t, rstate=1)
    statuses = [r["status"] for r in t.results]
    assert STATUS_FAIL in statuses and STATUS_OK in statuses and best["x"] <= 0.5


def test_parallel_trials_run_concurrently(tmp_path):
    peak, cur, lock = [0], [0], threading.Lock()

    def obj(p):
        with lock:
            cur[0] += 1
            peak[0] = max(peak[0], cur[0])
        time.sleep(0.05)
        with lock:
            cur[0] -= 1
        return p["x"] ** 2

    # threads: the objective counts its concurrency in this process ('auto' picks worker processes on a GPU machine)
    t = ParallelTrials(parallelism=4, executor="thread")
    fmin(obj, {"x": hp.uniform("x", -1, 1)}, algo=tpe.suggest, max_evals=16, trials=t, rstate=0)
    assert len(t) == 16 and 2 <= peak[0] <= 4


def test_trials_become_nested_child_runs(tmp_path):
    tracking.set_tracking_uri(str(tmp_path / "mlruns"))
    tracking.set_experiment("hpo")
    with tracking.start_run(run_name="hyperopt_tuning") as parent:
        fmin(lambda p: p["x"], {"x": hp.uniform("x", 0, 1)}, algo=rand.suggest, max_evals=5,
             trials=ParallelTrials(parallelism=2), rstate=0)
        pid = parent.info.run_id
    df = tracking.search_runs(filter_string=f'tags.mlflow.parentRunId = "{pid}"', order_by=["metrics.loss ASC"])
    assert len(df) == 5 and df["metrics.loss"].is_monotonic_increasing
    assert tracking.active_run() is None


def test_concurrent_trials_log_intact_child_runs(tmp_path):
    """SparkTrials(parallelism=4)-style use (reference P2/01:226): many trials logging at once must not interleave or lose
    records - every child run keeps its own parameters, its full metric history and its artifact, under the right parent."""
    import json
    import os

    tracking.set_tracking_uri(str(tmp_path / "mlruns"))
    tracking.set_experiment("hpo_stress")

    def obj(p):
        tag = f"{p['x']:.6f}"
        tracking.log_params({"x": tag, "twice": f"{2 * p['x']:.6f}"})
        for s in range(40):
            tracking.log_metric("curve", p["x"] + s, step=s)
        tracking.log_dict({"x": tag}, "who.json")
        time.sleep(0.01)
        return {"loss": p["x"] ** 2, "status": STATUS_OK}

    with tracking.start_run(run_name="parent") as parent:
        t = ParallelTrials(parallelism=8)
        fmin(obj, {"x": hp.uniform("x", -1, 1)}, algo=rand.suggest, max_evals=24, trials=t, rstate=3)
        pid = parent.info.run_id
    df = tracking.search_runs(filter_string=f'tags.mlflow.parentRunId = "{pid}"')
    assert len(df) == 24 and df["run_id"].is_unique
    for rid in df["run_id"]:
        r = tracking.get_run(rid)
        x = float(r.data.params["x"])
        assert abs(float(r.data.params["twice"]) - 2 * x) < 1e-5             # params of ONE trial, not a mixture
        hist = tracking.metric_history(rid, "curve")
        assert len(hist) == 40 and all(abs(v - (x + s)) < 1e-5 for s, v in enumerate(hist))   # history of ONE trial, in order
        assert abs(r.data.metrics["loss"] - x * x) < 1e-5
        with open(os.path.join(r.info.artifact_uri, "who.json")) as f:
            assert json.load(f)["x"] == r.data.params["x"]


def test_hyperopt_stopping_arguments():
    """`timeout`, `loss_threshold`, `early_stop_fn` (Hyperopt's fmin signature) stop the search; unknown Hyperopt keyword
    arguments are tolerated with a warning instead of a TypeError."""
    space = {"x": hp.uniform("x", -1, 1)}
    t = Trials()
    fmin(lambda p: (time.sleep(0.05), p["x"] ** 2)[1], space, algo=rand.suggest, max_evals=1000, trials=t, rstate=0, timeout=0.5)
    assert 2 <= len(t) < 60
    t = Trials()
    fmin(lambda p: p["x"] ** 2, space, algo=rand.suggest, max_evals=5000, trials=t, rstate=1, loss_threshold=1e-3)
    assert len(t) < 5000 and min(l for l in t.losses() if l is not None) <= 1e-3

    def no_progress(trials, best=None, stale=0):          # Hyperopt-style: stop after 5 trials without improvement
        cur = min(l for l in trials.losses() if l is not None)
        stale = 0 if best is None or cur < best else stale + 1
        return stale >= 5, [cur if best is None else min(best, cur), stale]

    t = Trials()
    fmin(lambda p: 1.0, space, algo=rand.suggest, max_evals=200, trials=t, rstate=2, early_stop_fn=no_progress)
    assert len(t) == 6                                      # first trial sets the best, five stale ones follow
    # threads: a 0.5 s budget is shorter than starting the worker processes 'auto' picks on a GPU machine
    t = ParallelTrials(parallelism=4, executor="thread")
    fmin(lambda p: (time.sleep(0.05), p["x"] ** 2)[1], space, algo=rand.suggest, max_evals=1000, trials=t, rstate=3, timeout=0.5)
    assert 4 <= len(t) < 120 and all(tr["result"].get("status") == STATUS_OK for tr in t.trials)
    with pytest.warns(UserWarning):
        fmin(lambda p: p["x"], space, algo=rand.suggest, max_evals=2, rstate=4, max_queue_len=4)


def _slot_objective(p):
    """Module-level objective for the process executor: reports which worker process / slot evaluated it."""
    import os
    import time

    from b200ddl import tracking

    time.sleep(0.15)
    tracking.log_metric("inner_metric", p["x"])
    return {"loss": (p["x"] - 0.3) ** 2, "status": hpo.STATUS_OK, "pid": os.getpid(),
            "slot": os.environ.get("B200DDL_TRIAL_SLOT"), "tid": hpo.current_trial()["tid"]}


def test_parallel_trials_process_executor(tmp_path):
    """`ParallelTrials(executor='process')`: trials run in persistent worker processes (one per slot), the objective
    travels by value, per-trial tracking lands in the trial's nested run, and a failing objective is recorded."""
    import os

    from b200ddl import tracking

    tracking.set_tracking_uri(str(tmp_path / "mlruns"))
    tracking.set_experiment("proc_hpo")
    trials = hpo.ParallelTrials(parallelism=3, executor="process")
    with tracking.start_run(run_name="parent") as parent:
        best = hpo.fmin(_slot_objective, {"x": hpo.hp.uniform("x", 0, 1)}, algo=hpo.rand.suggest, max_evals=9, trials=trials,
                        rstate=np.random.default_rng(0))
    assert 0 <= best["x"] <= 1 and len(trials) == 9
    pids = {t["result"]["pid"] for t in trials.trials}
    assert os.getpid() not in pids and 1 <= len(pids) <= 3            # evaluated in worker processes, reused across trials
    assert {t["result"]["slot"] for t in trials.trials} <= {"0", "1", "2"}
    assert sorted(t["result"]["tid"] for t in trials.trials) == list(range(9))
    kids = tracking.search_runs(filter_string=f"tags.mlflow.parentRunId = '{parent.info.run_id}'")
    assert len(kids) == 9 and kids["metrics.inner_metric"].notna().all()  # logged from inside the worker into the child run

    def flaky(p):
        if p["x"] > 0.5:
            raise ValueError("bad region")
        return p["x"]

    t2 = hpo.ParallelTrials(parallelism=2, executor="process")
    hpo.fmin(flaky, {"x": hpo.hp.uniform("x", 0, 1)}, algo=hpo.rand.suggest, max_evals=8, trials=t2,
             rstate=np.random.default_rng(1))
    states = [t["result"]["status"] for t in t2.trials]
    assert hpo.STATUS_FAIL in states and hpo.STATUS_OK in states
