"""Keras-like Trainer on CPU (BASELINE.json config 1: plumbing, world_size=1, no GPU)."""
import os

import numpy as np
import pytest
import torch

from b200ddl import optim, tracking
from b200ddl.models import build_model
from b200ddl.train import EarlyStopping, ModelCheckpoint, ReduceLROnPlateau, Trainer


def make_ds(batch=8, size=32, classes=5, seed=0):
    g = torch.Generator().manual_seed(seed)
    while True:
        y = torch.randint(0, classes, (batch,), generator=g)
        x = (torch.randint(0, 40, (batch, size, size, 3), generator=g) + (y * 40)[:, None, None, None]).clamp(0, 255)
        yield x.to(torch.uint8), y


def test_reference_model_only_head_is_trainable():
    m = build_model(224, 224, 3, 5, arch="mobilenetv2", device="cpu")   # the torch module, also where a GPU exists
    trainable = sum(p.numel() for p in m.parameters() if p.requires_grad)
    assert trainable == 1280 * 5 + 5 == 6405                       # SURVEY.md Q11 / P1/03:168-169
    assert build_model(0.3, arch="mobilenetv2", device="cpu").dropout.p == 0.3    # build_model(dropout) form (P2/01:92)


def test_fit_evaluate_predict_history_and_callbacks(tmp_path):
    model = build_model(32, 32, 3, 5, dropout=0.1, arch="mobilenetv2", freeze_base=False)
    tr = Trainer(model, device="cpu").compile(optimizer=optim.Adam(3e-3), loss="sparse_categorical_crossentropy",
                                              metrics=["accuracy"])
    ckpt = ModelCheckpoint(str(tmp_path / "ck" / "checkpoint-{epoch}.ckpt"), save_weights_only=True)
    hist = tr.fit(make_ds(), steps_per_epoch=12, epochs=3, verbose=0, validation_data=make_ds(seed=9),
                  validation_steps=3, callbacks=[ReduceLROnPlateau(monitor="val_loss", patience=10),
                                                 EarlyStopping(monitor="val_loss", min_delta=1e-2, patience=3), ckpt])
    assert set(hist.history) >= {"loss", "accuracy", "val_loss", "val_accuracy", "lr"}
    assert len(hist.history["val_loss"]) == 3 and hist.history["loss"][-1] < hist.history["loss"][0]
    assert [os.path.basename(p) for p in ckpt.saved] == ["checkpoint-1.ckpt", "checkpoint-2.ckpt", "checkpoint-3.ckpt"]
    loss, acc = tr.evaluate(make_ds(seed=3), steps=4)
    assert np.isfinite(loss) and 0 <= acc <= 1
    logits = tr.predict(np.random.randint(0, 255, (11, 32, 32, 3), dtype=np.uint8), batch_size=4)
    assert logits.shape == (11, 5)
    # checkpoint round trip
    before = tr.predict(np.zeros((2, 32, 32, 3), np.uint8))
    tr.load_weights(ckpt.saved[-1])
    assert np.allclose(before, tr.predict(np.zeros((2, 32, 32, 3), np.uint8)), atol=1e-5)


def test_early_stopping_stops():
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Flatten(), torch.nn.Linear(3 * 8 * 8, 5))
    tr = Trainer(model, device="cpu").compile(optimizer=optim.SGD(0.0))  # lr 0 => no improvement
    es = EarlyStopping(monitor="val_loss", min_delta=1e-2, patience=2)
    # A RE-ITERABLE validation set: like Keras, every validation pass starts from the beginning of the dataset, so
    # with validation_steps < len the same samples are scored each epoch and lr 0 gives a constant val_loss.  (A one-shot
    # generator would hand a different batch to every epoch and the stopping epoch would depend on luck.)
    gen = make_ds(size=8, seed=1)
    val = [next(gen) for _ in range(3)]
    hist = tr.fit(make_ds(size=8), steps_per_epoch=2, epochs=20, verbose=0, validation_data=val,
                  validation_steps=1, callbacks=[es])
    assert len(set(hist.history["val_loss"])) == 1          # same validation samples every epoch
    assert len(hist.history["loss"]) == 3 and es.stopped_epoch == 2


def test_autolog_and_model_reload(tmp_path):
    tracking.set_tracking_uri(str(tmp_path / "mlruns"))
    tracking.set_experiment("e")
    tracking.autolog()
    try:
        model = build_model(32, 32, 3, 5, arch="mobilenetv2", device="cpu")
        tr = Trainer(model, device="cpu").compile(optimizer=optim.Adam(1e-3))
        with tracking.start_run(run_name="single_node") as run:
            tr.fit(make_ds(), steps_per_epoch=2, epochs=2, verbose=0, validation_data=make_ds(seed=2), validation_steps=1)
            rid = run.info.run_id
    finally:
        tracking.autolog(disable=True)
    r = tracking.get_run(rid)
    assert r.data.params["epochs"] == "2" and "val_loss" in r.data.metrics
    assert tracking.metric_history(rid, "loss").__len__() == 2
    loaded = tracking.keras.load_model(f"runs:/{rid}/model")       # reference P1/03:438
    x = np.random.randint(0, 255, (3, 32, 32, 3), dtype=np.uint8)
    assert np.allclose(loaded.predict(x, batch_size=3), tr.predict(x, batch_size=3), atol=1e-4)
    assert "Trainable params: 6,405" in loaded.summary()


def test_optimizer_lookup_by_name():
    assert optim.get("Adam") is optim.Adam and optim.get("Adadelta") is optim.Adadelta   # reference P2/01:154
    with pytest.raises(ValueError):
        optim.get("Nope")


def test_save_load_resume_continues_training(tmp_path):
    """Checkpoint / resume (SURVEY.md 5.4): `save()` after two epochs, a NEW trainer `load()`s it and continues with
    `initial_epoch=2`; weights, optimizer moments and the step counter carry over, so the resumed run is the same run."""
    def make(lr=3e-3):
        torch.manual_seed(1)
        model = build_model(32, 32, 3, 5, dropout=0.0, arch="mobilenetv2", freeze_base=False)
        return Trainer(model, device="cpu").compile(optimizer=optim.Adam(lr), loss="sparse_categorical_crossentropy",
                                                    metrics=["accuracy"])

    # uninterrupted reference: 4 epochs over a deterministic stream
    ref = make()
    h_ref = ref.fit(make_ds(seed=4), steps_per_epoch=6, epochs=4, verbose=0)
    # interrupted: 2 epochs, save, new process-equivalent trainer, load, 2 more epochs over the rest of the stream
    a = make()
    stream = make_ds(seed=4)
    h_a = a.fit(stream, steps_per_epoch=6, epochs=2, verbose=0)
    path = str(tmp_path / "resume.pt")
    a.save(path)
    b = make(lr=1.0)                      # wrong LR on purpose: load() must restore the saved one
    b.load(path)
    opt_b = b.optimizer
    assert opt_b.t == 12 and abs(opt_b.learning_rate - 3e-3) < 1e-12
    h_b = b.fit(stream, steps_per_epoch=6, epochs=4, initial_epoch=2, verbose=0)
    assert len(h_b.history["loss"]) == 2                               # epochs 3 and 4 only
    assert np.allclose(h_a.history["loss"], h_ref.history["loss"][:2], rtol=1e-4)
    assert np.allclose(h_b.history["loss"], h_ref.history["loss"][2:], rtol=2e-3), (h_b.history["loss"], h_ref.history["loss"])
    # weights-only files (ModelCheckpoint / save_weights) load through the same entry point
    a.save_weights(str(tmp_path / "w.pt"))
    c = make()
    c.load(str(tmp_path / "w.pt"))
    x = np.zeros((2, 32, 32, 3), np.uint8)
    assert np.allclose(a.predict(x), c.predict(x), atol=1e-5)
    # optimizer mismatch is an error, not silent garbage
    d = Trainer(build_model(32, 32, 3, 5, arch="mobilenetv2", device="cpu"), device="cpu").compile(optimizer=optim.SGD(0.1))
    with pytest.raises(ValueError):
        d.load(path)


def test_compile_with_keras_style_loss_object():
    """The reference's spelling: `loss=SparseCategoricalCrossentropy(from_logits=True)`, `metrics=['accuracy']`."""
    from b200ddl.train import losses

    model = torch.nn.Sequential(torch.nn.Flatten(), torch.nn.Linear(3 * 8 * 8, 5))
    tr = Trainer(model, device="cpu").compile(optimizer=optim.Adam(learning_rate=1e-2),
                                              loss=losses.SparseCategoricalCrossentropy(from_logits=True), metrics=["accuracy"])
    h = tr.fit(make_ds(size=8), steps_per_epoch=4, epochs=2, verbose=0)
    assert set(h.history) >= {"loss", "accuracy"}
    with pytest.raises(ValueError):
        losses.SparseCategoricalCrossentropy()                 # probabilities are not what the models output
    with pytest.raises(ValueError):
        Trainer(model, device="cpu").compile(optimizer=optim.SGD(0.1), loss="mse")
