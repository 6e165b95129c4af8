"""use_ring models on the structure routes: the host route against ``predict_structures(..., ring_aromatic=)`` and
``DeviceDataIterator.from_structures(..., use_ring=True, ring_aromatic=)`` on one GPU.

Workloads (seeded weights, targets and flags):
- ptgp: PtGP-like structures (tests/test_ring_routes.py ``ptgp_like``: graphene sheet + Pt cluster, 172-253 sites;
  carbon [1, 1], Pt [0, 0], random flags in every third structure) under the shipped PtGP config (11 layers,
  g_update=False with gaussian_d=4.0, batch 64); structures with a Voronoi cell beyond the cell search's capacity are
  dropped and counted;
- qm9_ring: QM9-like boxed molecules with random 0/1 flags under the QM9 config with use_ring=True (7 layers, batch
  128).
Reported, with the card's name and power limit read in the same run:
- structures/s of the host route (compute_voronoi_neighbors -> DataIterator(use_ring=True).csr_item -> predict, on the
  shape classes predict_structures uses) and of predict_structures, each after a warm-up pass, in windows of >= 1 s
  ending in a device synchronise; max |diff| of the two routes' outputs;
- epoch time through ``fit`` (default mode, Dropout and shuffle on) for the host DataIterator(use_ring=True) and for
  DeviceDataIterator.from_structures of the same structures and flags: one warm-up epoch, then the mean of two timed
  epochs; and the ceiling of the device route, steps x the CUDA-graph replay time of each batch's step (CUDA events),
  as tools/device_data_bench.py does.

    python tools/ring_routes_bench.py [--out profiles/r03_ring_routes.log]
"""
from __future__ import annotations

import argparse
import os
import re
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from structure_predict_bench import rate                    # noqa: E402
from tests.test_ring_routes import ptgp_like, ring_rows     # noqa: E402
from tests.test_voronoi import molecule                     # noqa: E402
from voronoi_bench import card                              # noqa: E402


def within_capacity(structs, flags):
    """Drop the structures with a Voronoi cell beyond the cell search's capacity (64 facets: a Pt atom with few cluster
    neighbours can meet more carbons of the two sheets), which every route refuses; returns the rest and the count."""
    from scann_b200 import voronoi as V
    dropped = 0
    while True:
        try:
            V.voronoi_polyhedra(structs)
            return structs, flags, dropped
        except ValueError as e:
            m = re.match(r"structure (\d+), site \d+: its Voronoi cell exceeds the kernel's capacity", str(e))
            if m is None:
                raise
            k = int(m.group(1))
            structs, flags, dropped = structs[:k] + structs[k + 1:], flags[:k] + flags[k + 1:], dropped + 1


def workload(name, n, seed=0):
    """(structs, flags, targets, config name, config overrides, batch size, structures dropped)."""
    dropped = 0
    if name == "ptgp":
        structs, flags, dropped = within_capacity(*ptgp_like(n, seed=seed))
        n = len(structs)
        cfg_name, over, bs = "ptgp", {"g_update": False, "gaussian_d": 4.0}, 64
    else:
        rng = np.random.default_rng(seed)
        structs = [molecule(rng, int(rng.integers(9, 30))) for _ in range(n)]
        flags = [rng.integers(0, 2, (len(s.atomic_numbers), 2)) for s in structs]
        cfg_name, over, bs = "qm9", {}, 128
    y = np.random.default_rng(seed + 1).standard_normal(n).tolist()
    return structs, flags, y, cfg_name, over, bs, dropped


def model(cfg_name, over, infer):
    from scann_b200.config import model_spec
    from scann_b200.configs import get_config
    from scann_b200.model import create_model
    from scann_b200.params import ParamLayout
    cfg = get_config(cfg_name)
    cfg["model"].update(use_ring=True, **over)
    return create_model(cfg, infer=infer, arena=ParamLayout(model_spec(cfg)).randomize_arena(3))


def predict_rates(name, n, lines):
    import torch
    from scann_b200 import voronoi as V
    from scann_b200.datagenerator import DataIterator
    from scann_b200.model import shape_class
    structs, flags, _, cfg_name, over, bs, dropped = workload(name, n)
    m = model(cfg_name, over, infer=True)
    angle = bool(m.spec.g_update)
    S, atoms = len(structs), sum(len(s.atomic_numbers) for s in structs)

    def host_route():
        de, dn = ring_rows(structs, V.compute_voronoi_neighbors(structs), flags)
        it = DataIterator(de, dn, batch_size=bs, g_update=angle, use_ring=True)
        ys, gas = [], []
        for i in range(len(it)):
            csr, _ = it.csr_item(i)
            csr["M"], csr["N"] = shape_class(csr["M"], csr["N"])
            y, ga = m.predict(csr)
            ys.append(y)
            gas.extend(ga[k, :c, 0] for k, c in enumerate(np.diff(csr["struct_atom_off"])))
        return np.concatenate(ys), gas

    def device_route():
        return m.predict_structures(structs, batch_size=bs, ring_aromatic=flags)

    reps_h, t_h = rate(host_route)
    reps_d, t_d = rate(device_route)
    torch.cuda.synchronize()
    (y_h, ga_h), (y_d, ga_d) = host_route(), device_route()
    dy = float(np.abs(y_h.astype(np.float64) - y_d).max())
    dga = max(float(np.abs(g.astype(np.float64) - h).max()) for g, h in zip(ga_d, ga_h))
    h_rate, d_rate = reps_h * S / t_h, reps_d * S / t_d
    lines.append(f"{name} predict: {S} structures ({dropped} of {S + dropped} dropped: a cell beyond the capacity), "
                 f"{atoms} atoms, {cfg_name} config with use_ring "
                 f"(L{m.spec.n_attention}), batch {bs}; host route {h_rate:,.0f} structures/s ({reps_h} passes in "
                 f"{t_h:.2f} s); predict_structures(ring_aromatic=) {d_rate:,.0f} structures/s ({reps_d} passes in "
                 f"{t_d:.2f} s), {d_rate / h_rate:.1f}x; max |diff| y {dy:.1e}, ga {dga:.1e}")
    print(lines[-1], flush=True)


def epoch_times(name, n, lines):
    import torch
    from scann_b200 import voronoi as V
    from scann_b200.datagenerator import DataIterator, DeviceDataIterator
    structs, flags, y, cfg_name, over, bs, dropped = workload(name, n, seed=5)
    n = len(structs)
    g = bool(over.get("g_update", True))
    t0 = time.perf_counter()
    de, dn = ring_rows(structs, V.compute_voronoi_neighbors(structs), flags, y)
    np.random.seed(0)
    host = DataIterator(de, dn, batch_size=bs, shuffle=True, g_update=g, use_ring=True)
    t_build_h = time.perf_counter() - t0
    t0 = time.perf_counter()
    np.random.seed(0)
    dev = DeviceDataIterator.from_structures(structs, y, batch_size=bs, shuffle=True, g_update=g, use_ring=True,
                                             ring_aromatic=flags)
    torch.cuda.synchronize()
    t_build_d = time.perf_counter() - t0
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

    m_h, m_d = model(cfg_name, over, False), model(cfg_name, over, False)
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
    lines.append(
        f"{name} fit: {n} structures ({dropped} dropped: a cell beyond the capacity), {cfg_name} config with use_ring (L{m_d.spec.n_attention}), batch {bs}, {steps} "
        f"steps per epoch\n"
        f"  data-set build: compute_voronoi_neighbors + DataIterator {t_build_h:.2f} s; "
        f"DeviceDataIterator.from_structures {t_build_d:.2f} s\n"
        f"  epoch through fit (Dropout, shuffle): host DataIterator {1e3 * t_h:.1f} ms ({1e3 * t_h / steps:.3f} ms/step); "
        f"DeviceDataIterator {1e3 * t_d:.1f} ms ({1e3 * t_d / steps:.3f} ms/step)\n"
        f"  ceiling: {steps} steps x graph-replay step time = {1e3 * t_ceil:.1f} ms ({1e3 * t_ceil / steps:.3f} ms/step); "
        f"device route {100 * (t_d / t_ceil - 1):+.1f} %, host route {100 * (t_h / t_ceil - 1):+.1f} % of it")
    print(lines[-1], flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-ptgp", type=int, default=512)
    ap.add_argument("--n-qm9", type=int, default=4096)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    lines = [f"card: {card()}", f"torch {torch.__version__}, device {torch.cuda.get_device_name(0)}"]
    predict_rates("ptgp", a.n_ptgp, lines)
    predict_rates("qm9_ring", a.n_qm9, lines)
    epoch_times("ptgp", a.n_ptgp, lines)
    epoch_times("qm9_ring", 2 * a.n_qm9, lines)
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
