"""Host-side training shell: callbacks of scann_b200/callbacks.py against the behaviour of the Keras callbacks and
of the reference's SGDRC (scann/layers/custom_layers.py:78-179) that they restate."""
import math

import numpy as np

from scann_b200 import callbacks as C


class FakeModel:
    def __init__(self):
        self.lr, self.stop_training, self.saved = 1e-3, False, []

    def _lr_now(self):
        return self.lr

    def save(self, path):
        self.saved.append(("full", path))

    def save_weights(self, path):
        self.saved.append(("weights", path))


def test_sgdrc_schedule_matches_the_reference_state_machine():
    s = C.SGDRC(lr_min=1e-4, lr_max=5e-4, t0=3, tmult=2, lr_max_compression=1.2, trigger_val_mae=0.5, show_lr=False)
    s.on_train_begin({})
    lrs = []
    val = [0.9, 0.7, 0.45, 0.44, 0.46, 0.43, 0.42, 0.41, 0.40, 0.39, 0.38]
    for ep, v in enumerate(val):
        lrs.append(s.lr_scheduler(ep))
        s.on_epoch_end(ep, {"val_mae": v})
    # not triggered for the first three epochs (trigger seen at the end of epoch 2): constant lr_max
    assert lrs[:3] == [5e-4, 5e-4, 5e-4]
    # epoch 3: tcur 2 of ti 3 -> cosine position 2/3 with peak 5e-4
    cos = lambda peak, t, ti: 1e-4 + (peak - 1e-4) * (1 + math.cos(math.pi * t / ti)) / 2
    assert lrs[3] == cos(5e-4, 2, 3)
    assert lrs[4] == cos(5e-4, 3, 3) == 1e-4
    # cycle ends: length 3 -> 6, peak = next warm-up = max(5e-4 / 1.2, lr at the last improvement)
    peak2 = max(5e-4 / 1.2, lrs[3])
    assert abs(lrs[5] - cos(peak2, 1, 6)) < 1e-18
    assert all(abs(lrs[5 + k] - cos(peak2, 1 + k, 6)) < 1e-18 for k in range(6))
    assert min(lrs) >= 1e-4 - 1e-18 and max(lrs) <= 5e-4


def test_checkpoint_and_early_stopping(tmp_path):
    m = FakeModel()
    ck = C.ModelCheckpoint(str(tmp_path / "models" / "model_{epoch}.h5"), monitor="val_mae", save_best_only=True)
    es = C.EarlyStopping(monitor="val_mae", patience=2)
    for cb in (ck, es):
        cb.set_model(m)
        cb.on_train_begin({})
    vals = [0.5, 0.4, 0.45, 0.41, 0.42]
    stopped = None
    for ep, v in enumerate(vals):
        for cb in (ck, es):
            cb.on_epoch_end(ep, {"val_mae": v})
        if m.stop_training:
            stopped = ep
            break
    assert [p for _, p in m.saved] == [str(tmp_path / "models" / f"model_{e}.h5") for e in (1, 2)]
    assert all(kind == "full" for kind, _ in m.saved)
    assert stopped == 3                                  # two epochs without improvement after the best (0.4)


def test_learning_rate_scheduler_sets_the_model_rate():
    m = FakeModel()
    sch = C.LearningRateScheduler(lambda ep: 1e-3 * 0.5 ** ep)
    sch.set_model(m)
    logs = {}
    sch.on_epoch_begin(2)
    sch.on_epoch_end(2, logs)
    assert m.lr == 2.5e-4 and logs["lr"] == 2.5e-4
