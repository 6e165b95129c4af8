"""Training input: the host route (``DataIterator``) against the device-resident data set (``DeviceDataIterator``).

Workloads are the generators of tools/voronoi_bench.py (tests/test_voronoi.py): QM9-like boxed molecules under the
QM9 config (7 layers, batch 128) and MP2018-like crystals under the MP2018 config (9 layers, batch 64), seeded weights,
seeded targets.  Per workload, on one GPU, the card's name and power limit read in the same run:
- data-set build: compute_voronoi_neighbors + DataIterator against DeviceDataIterator.from_structures;
- epoch time through ``fit`` (default mode, Dropout and shuffle on) for both iterators over the same data: one warm-up
  epoch, then the mean of two timed epochs, each ending in a device synchronise;
- the ceiling of the device route: the steps of one epoch x the CUDA-graph replay time of each batch's train step,
  measured with CUDA events on the same shapes;
- one validation pass (a tenth of the data set) through each route;
- ``DataIterator.csr_item`` per batch (host clock over an epoch) and ``scann_gather_batch`` per batch (a CUDA-event
  pair around each launch, every batch of an epoch, 20 rounds);
- a deterministic-mode check on the first 1024 structures (2 epochs with a validation set): both routes give the same
  History and the same parameter bits (skipped where a batch has more than 32 neighbours per atom, which the
  deterministic mode refuses).

    python tools/device_data_bench.py [--qm9 16384] [--mp 8192] [--out profiles/r03_device_data.log]
"""
from __future__ import annotations

import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from tests.test_voronoi import molecule, random_cell     # noqa: E402
from voronoi_bench import card                            # noqa: E402

CONFIGS = {"qm9_boxed": ("qm9", 128), "mp2018_crystal": ("mp2018", 64)}


def host_iterator(structs, lists, y, bs, g_update, shuffle):
    from scann_b200.datagenerator import DataIterator
    S = len(structs)
    de, dn = np.empty(S, object), np.empty(S, object)
    for k, (s, nb) in enumerate(zip(structs, lists)):
        de[k], dn[k] = (list(s.atomic_numbers), float(y[k])), nb
    return DataIterator(de, dn, batch_size=bs, g_update=g_update, shuffle=shuffle)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qm9", type=int, default=16384)
    ap.add_argument("--mp", type=int, default=8192)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    from scann_b200 import voronoi as V
    from scann_b200.configs import get_config
    from scann_b200.datagenerator import DeviceDataIterator
    from scann_b200.model import _batch_errors, create_model

    lines = [f"card: {card()}", f"torch {torch.__version__}, device {torch.cuda.get_device_name(0)}"]
    sizes = {"qm9_boxed": a.qm9, "mp2018_crystal": a.mp}
    for name in ("qm9_boxed", "mp2018_crystal"):
        rng = np.random.default_rng(0)
        structs = ([molecule(rng, int(rng.integers(9, 30))) for _ in range(sizes[name])] if name == "qm9_boxed" else
                   [random_cell(rng, int(rng.integers(2, 65))) for _ in range(sizes[name])])
        cfg_name, bs = CONFIGS[name]
        cfg = get_config(cfg_name)
        S = len(structs)
        y = np.random.default_rng(1).standard_normal(S)
        n_val = S // 10
        g_update = bool(cfg["model"]["g_update"])
        DeviceDataIterator.from_structures(structs[:64], y[:64], batch_size=bs, g_update=g_update)   # warm-up

        # ---- data-set build
        t0 = time.perf_counter()
        lists = V.compute_voronoi_neighbors(structs)
        np.random.seed(0)
        host = host_iterator(structs[n_val:], lists[n_val:], y[n_val:], bs, g_update, True)
        host_val = host_iterator(structs[:n_val], lists[:n_val], y[:n_val], bs, g_update, False)
        t_build_h = time.perf_counter() - t0
        t0 = time.perf_counter()
        np.random.seed(0)
        dev = DeviceDataIterator.from_structures(structs[n_val:], y[n_val:], batch_size=bs, shuffle=True,
                                                 g_update=g_update)
        dev_val = DeviceDataIterator.from_structures(structs[:n_val], y[:n_val], batch_size=bs, g_update=g_update)
        torch.cuda.synchronize()
        t_build_d = time.perf_counter() - t0
        steps = len(host)

        # ---- csr_item per batch (host clock)
        t0 = time.perf_counter()
        for i in range(steps):
            host.csr_item(i)
        csr_ms = 1e3 * (time.perf_counter() - t0) / steps

        # ---- epoch time through fit
        def epoch_times(it, model):
            model.fit(it, epochs=1, verbose=0)           # warm-up: shape classes, graphs
            torch.cuda.synchronize()
            c0, ts = model.engine.graph_captures, []
            for _ in range(2):
                t = time.perf_counter()
                model.fit(it, epochs=1, verbose=0)
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t)
            return float(np.mean(ts)), model.engine.graph_captures - c0

        m_h, m_d = create_model(cfg, seed=3), create_model(cfg, seed=3)
        t_ep_h, cap_h = epoch_times(host, m_h)
        t_ep_d, cap_d = epoch_times(dev, m_d)

        # ---- ceiling: steps x graph-replay train-step time of the same shapes (CUDA events)
        eng = m_d.engine
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for i in range(steps):
            b = eng.load_batch_gather(dev, *dev.batch_shape(i), plan=False)
            eng.train_step(b, b.target, 1e-4, replan=True)
            ev[i][0].record()
            for _ in range(3):
                eng.train_step(b, b.target, 1e-4, replan=True)
            ev[i][1].record()
        torch.cuda.synchronize()
        t_ceiling = sum(e0.elapsed_time(e1) for e0, e1 in ev) / 3 / 1e3

        # ---- scann_gather_batch per batch (a CUDA-event pair around each launch, 20 rounds over the epoch's batches)
        shapes = [dev.batch_shape(i) for i in range(steps)]
        for sh in shapes:
            eng.load_batch_gather(dev, *sh, plan=False)
        eng.prof = {}
        for _ in range(20):
            for sh in shapes:
                eng.load_batch_gather(dev, *sh, plan=False)
        torch.cuda.synchronize()
        n_gather, gather_ms = eng.prof_summary()["gather_batch"]
        eng.prof = None
        gather_us = 1e3 * gather_ms

        # ---- one validation pass per route
        def val_host():
            return [m_h.evaluate_batch(*host_val[i]) for i in range(len(host_val))]

        def val_dev():
            return [_batch_errors(*m_d.predict_device_batch(dev_val, i)) for i in range(len(dev_val))]
        val_host(), val_dev()
        t0 = time.perf_counter()
        val_host()
        t_val_h = time.perf_counter() - t0
        t0 = time.perf_counter()
        val_dev()
        t_val_d = time.perf_counter() - t0

        # ---- deterministic mode: both routes, same bits
        def det(route):
            n = min(1024, S - n_val)
            np.random.seed(5)
            it = host_iterator(structs[n_val:n_val + n], lists[n_val:n_val + n], y[n_val:n_val + n], bs, g_update, True)
            vit = host_iterator(structs[:n_val], lists[:n_val], y[:n_val], bs, g_update, False)
            if route == "device":
                it, vit = DeviceDataIterator.from_data_iterator(it), DeviceDataIterator.from_data_iterator(vit)
            m = create_model(cfg, seed=3, deterministic=True)
            h = m.fit(it, epochs=2, validation_data=vit, verbose=0).history
            return h, m.engine.params.cpu().numpy()
        try:
            (hh, ph), (hd, pd) = det("host"), det("device")
            same = hh == hd and np.array_equal(ph.view(np.uint32), pd.view(np.uint32))
            det_txt = f"deterministic check (2 epochs, {min(1024, S - n_val)} structures): History and parameters " \
                      f"{'identical' if same else 'DIFFER'} (loss {hh['loss'][-1]:.6f} / {hd['loss'][-1]:.6f})"
        except NotImplementedError as e:
            det_txt = f"deterministic check: not applicable ({e})"

        atoms = sum(len(s.cart_coords) for s in structs)
        lines.append(
            f"{name}: {S} structures ({S - n_val} train, {n_val} validation), {atoms} atoms, {cfg_name} config "
            f"(L{cfg['model']['n_attention']}), batch {bs}, {steps} steps per epoch\n"
            f"  data-set build: compute_voronoi_neighbors + DataIterator {t_build_h:.2f} s; "
            f"DeviceDataIterator.from_structures {t_build_d:.2f} s ({t_build_h / t_build_d:.1f}x)\n"
            f"  epoch through fit (Dropout, shuffle): host DataIterator {1e3 * t_ep_h:.1f} ms "
            f"({1e3 * t_ep_h / steps:.3f} ms/step, {cap_h} graph captures in the timed epochs); DeviceDataIterator "
            f"{1e3 * t_ep_d:.1f} ms ({1e3 * t_ep_d / steps:.3f} ms/step, {cap_d} captures)\n"
            f"  ceiling: {steps} steps x graph-replay step time = {1e3 * t_ceiling:.1f} ms "
            f"({1e3 * t_ceiling / steps:.3f} ms/step); device route {100 * (t_ep_d / t_ceiling - 1):+.1f} %, "
            f"host route {100 * (t_ep_h / t_ceiling - 1):+.1f} % of it\n"
            f"  validation pass ({len(host_val)} batches): host (padded __getitem__ + predict) {1e3 * t_val_h:.1f} ms; "
            f"device (gather + predict_step) {1e3 * t_val_d:.1f} ms\n"
            f"  DataIterator.csr_item {csr_ms:.3f} ms per batch (host clock, one epoch); scann_gather_batch "
            f"{gather_us:.2f} us per batch (CUDA events around each of {n_gather} launches)\n"
            f"  {det_txt}")
        print(lines[-1], flush=True)
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
