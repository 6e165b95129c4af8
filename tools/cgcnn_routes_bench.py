"""feature='cgcnn' models: the padded feature-vector route (host ``DataIterator``, ``[B, M, 92]`` per step) against the
table route (atomic numbers embedded through the per-element table on the device: ``DeviceDataIterator``,
``predict_structures``).

Workload: QM9-like boxed molecules (tests/test_voronoi.py generators) under the QM9 config with feature='cgcnn'
(7 layers, batch 128), seeded weights and targets, the 100-row stand-in table of ``synth.cgcnn_table``.  On one GPU,
with the card's name and power limit read in the same run:
- epoch time through ``fit`` (default mode, Dropout and shuffle on) for the host DataIterator and for
  DeviceDataIterator.from_data_iterator of it: one warm-up epoch, then the mean of two timed epochs, each ending in a
  device synchronise; and the ceiling of the device route, steps x the CUDA-graph replay time of each batch's step
  (CUDA events);
- structures per second through ``predict_structures(..., atomic_features=T)`` against the host route
  (compute_voronoi_neighbors + DataIterator(feature='cgcnn') + ``predict`` of each padded batch), after a warm-up pass;
- ``--profile`` (a separate run): device time per train step of the embedding kernels of each route (eager launches,
  torch.profiler with CUDA activities over 20 steps of the same batch).

    python tools/cgcnn_routes_bench.py [--n 8192] [--out profiles/r03_cgcnn_routes.log] [--profile]
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

from tests.test_voronoi import molecule                    # noqa: E402
from voronoi_bench import card                              # noqa: E402

# embedding kernels of the two routes (forward and backward); everything else of the step is shared
EMBED_KERNELS = ("small_dense_fwd_kernel", "embed_fwd_kernel", "embed_bwd_rows_kernel", "embed_bwd_cols_kernel",
                 "embed_bwd_gather_kernel", "embed_bwd_final_kernel", "cgcnn_table_bwd_kernel")


def data(n, seed=0):
    from scann_b200 import voronoi as V
    from scann_b200.synth import cgcnn_table
    rng = np.random.default_rng(seed)
    structs = [molecule(rng, int(rng.integers(9, 30))) for _ in range(n)]
    y = np.random.default_rng(1).standard_normal(n)
    lists = V.compute_voronoi_neighbors(structs)
    de, dn = np.empty(n, object), np.empty(n, object)
    for k, (s, nb) in enumerate(zip(structs, lists)):
        de[k], dn[k] = (list(s.atomic_numbers), float(y[k])), nb
    return structs, de, dn, cgcnn_table()


def model(infer=False):
    from scann_b200.configs import get_config
    from scann_b200.model import create_model
    cfg = get_config("qm9", feature="cgcnn")
    return create_model(cfg, seed=3, infer=infer), cfg


def timing(a, lines):
    import torch
    from scann_b200.datagenerator import DataIterator, DeviceDataIterator
    structs, de, dn, T = data(a.n)
    np.random.seed(0)
    host = DataIterator(de, dn, batch_size=128, shuffle=True, feature="cgcnn", atomic_features=T, g_update=True)
    dev = DeviceDataIterator.from_data_iterator(host)
    steps = len(host)

    def epochs(it, m):
        m.fit(it, epochs=1, verbose=0)
        torch.cuda.synchronize()
        ts = []
        for _ in range(2):
            t = time.perf_counter()
            m.fit(it, epochs=1, verbose=0)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t)
        return float(np.mean(ts))

    (m_h, cfg), (m_d, _) = model(), model()
    t_h, t_d = epochs(host, m_h), epochs(dev, m_d)
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
    t_ceil = sum(e0.elapsed_time(e1) for e0, e1 in ev) / 3 / 1e3

    # ---- predict_structures against the host route
    from scann_b200 import voronoi as V
    mi, _ = model(infer=True)
    sub = structs[:a.n_predict]

    def host_route():
        lists = V.compute_voronoi_neighbors(sub)
        de_p, dn_p = np.empty(len(sub), object), np.empty(len(sub), object)
        for k, (s, nb) in enumerate(zip(sub, lists)):
            de_p[k], dn_p[k] = (list(s.atomic_numbers), 0.0), nb
        it = DataIterator(de_p, dn_p, batch_size=128, feature="cgcnn", atomic_features=T, g_update=True)
        return [mi.predict(it[i][0]) for i in range(len(it))]

    def dev_route():
        return mi.predict_structures(sub, batch_size=128, atomic_features=T)

    rates = {}
    for name, fn in (("host", host_route), ("device", dev_route)):
        fn()
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        rates[name] = len(sub) / (time.perf_counter() - t)
    lines.append(
        f"qm9_boxed cgcnn: {a.n} structures, qm9 config with feature='cgcnn' (L{cfg['model']['n_attention']}), batch 128, "
        f"{steps} steps per epoch, table {T.shape[0]} x 92\n"
        f"  epoch through fit (Dropout, shuffle): host DataIterator (padded [B, M, 92] route) {1e3 * t_h:.1f} ms "
        f"({1e3 * t_h / steps:.3f} ms/step); DeviceDataIterator (table route) {1e3 * t_d:.1f} ms "
        f"({1e3 * t_d / steps:.3f} ms/step)\n"
        f"  ceiling: {steps} steps x graph-replay step time of the table route = {1e3 * t_ceil:.1f} ms "
        f"({1e3 * t_ceil / steps:.3f} ms/step); device route {100 * (t_d / t_ceil - 1):+.1f} %, "
        f"host route {100 * (t_h / t_ceil - 1):+.1f} % of it\n"
        f"  predict, {len(sub)} structures, batch 128: compute_voronoi_neighbors + DataIterator + predict "
        f"{rates['host']:.0f} structures/s; predict_structures(atomic_features=T) {rates['device']:.0f} structures/s "
        f"({rates['device'] / rates['host']:.1f}x)")


def profile(a, lines):
    import torch
    from torch.profiler import ProfilerActivity
    from scann_b200.datagenerator import DataIterator, DeviceDataIterator
    _, de, dn, T = data(256)
    host = DataIterator(de, dn, batch_size=128, feature="cgcnn", atomic_features=T, g_update=True)
    dev = DeviceDataIterator.from_data_iterator(host)
    out = {}
    for route in ("padded", "table"):
        m, _ = model()
        eng = m.engine
        eng.use_graphs = False                  # eager launches: every kernel is its own trace record
        eng.train_dropout = True
        if route == "table":
            eng.set_atomic_features(T)
            b = eng.load_batch_gather(dev, *dev.batch_shape(0), plan=False)
            target = b.target
        else:
            inputs, target = host[0]
            b = eng.load_batch(inputs, plan=False)
        for _ in range(3):
            eng.train_step(b, target, 1e-4, replan=True)
        torch.cuda.synchronize()
        n = 20
        with torch.profiler.profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n):
                eng.train_step(b, target, 1e-4, replan=True)
            torch.cuda.synchronize()
        per = {}
        for e in prof.key_averages():
            if any(e.key.startswith(k) or k in e.key for k in EMBED_KERNELS):
                us = getattr(e, "device_time_total", None)
                us = e.cuda_time_total if us is None else us
                per[e.key.split("(")[0]] = us / n
        out[route] = per
    for route, per in out.items():
        lines.append(f"  embedding kernels per train step, {route} route (torch.profiler, 20 eager steps, batch 0 of "
                     f"the 256-molecule set): {sum(per.values()):.1f} us in all; " +
                     ", ".join(f"{k} {v:.1f} us" for k, v in sorted(per.items())))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=8192)
    ap.add_argument("--n-predict", type=int, default=4096)
    ap.add_argument("--out", default="")
    ap.add_argument("--profile", action="store_true")
    a = ap.parse_args()
    import torch
    lines = [f"card: {card()}", f"torch {torch.__version__}, device {torch.cuda.get_device_name(0)}"]
    (profile if a.profile else timing)(a, lines)
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a" if a.profile else "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
