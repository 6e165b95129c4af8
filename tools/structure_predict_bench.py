"""Structures -> predictions: the host route against ``predict_structures`` on one GPU.

Workloads are the generators of tools/voronoi_bench.py: QM9-like boxed molecules under the QM9 config (7 layers,
batch 128) and MP2018-like crystals under the MP2018 config (9 layers, batch 64), seeded weights.  Reports
- structures/s of the host route: compute_voronoi_neighbors -> DataIterator.csr_item -> predict, on the padded shapes
  predict_structures uses (so both routes replay the same CUDA graphs and only the neighbour-list step differs);
- structures/s of predict_structures;
- CUDA-event time per structure of scann_voronoi_neighbors (all retry passes), of scann_voronoi_select +
  scann_voronoi_batch_csr, and of the model (pack + plan + forward) -- one instrumented pass, outside the timed windows;
- max |diff| between the two routes' outputs.
Every shape is warmed up first; timed windows are >= 1 s and end in a device synchronise.

    python tools/structure_predict_bench.py [--n 2000] [--out profiles/r03_predict_structures.log]
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

from voronoi_bench import card, workloads        # noqa: E402

CONFIGS = {"qm9_boxed": ("qm9", 128), "mp2018_crystal": ("mp2018", 64)}


def rate(fn, min_s=1.0):
    fn()                                        # warm-up: every shape class of the workload
    reps, t = 0, 0.0
    t0 = time.perf_counter()
    while t < min_s:
        fn()
        reps += 1
        t = time.perf_counter() - t0
    return reps, t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=2000)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    from scann_b200 import voronoi as V
    from scann_b200.config import model_spec
    from scann_b200.configs import get_config
    from scann_b200.datagenerator import DataIterator
    from scann_b200.model import create_model, shape_class
    from scann_b200.params import ParamLayout

    lines = [f"card: {card()}", f"torch {torch.__version__}, device {torch.cuda.get_device_name(0)}"]
    for name, structs in workloads(a.n).items():
        cfg_name, bs = CONFIGS[name]
        cfg = get_config(cfg_name)
        model = create_model(cfg, infer=True, arena=ParamLayout(model_spec(cfg)).randomize_arena(3))
        angle = bool(model.spec.g_update)
        S = len(structs)
        atoms = sum(len(s.cart_coords) for s in structs)

        def host_route():
            lists = V.compute_voronoi_neighbors(structs)
            de, dn = np.empty(S, object), np.empty(S, object)
            for k, (s, nb) in enumerate(zip(structs, lists)):
                de[k], dn[k] = (list(s.atomic_numbers), 0.0), nb
            it = DataIterator(de, dn, batch_size=bs, g_update=angle)
            ys, gas = [], []
            for i in range(len(it)):
                csr, _ = it.csr_item(i)
                csr["M"], csr["N"] = shape_class(csr["M"], csr["N"])
                y, ga = model.predict(csr)
                ys.append(y)
                gas.extend(ga[k, :n, 0] for k, n in enumerate(np.diff(csr["struct_atom_off"])))
            return np.concatenate(ys), gas

        def device_route():
            return model.predict_structures(structs, batch_size=bs)

        reps_h, t_h = rate(host_route)
        reps_d, t_d = rate(device_route)
        y_h, ga_h = host_route()
        y_d, ga_d = device_route()
        dy = float(np.abs(y_h.astype(np.float64) - y_d).max())
        dga = max(float(np.abs(g.astype(np.float64) - h).max()) for g, h in zip(ga_d, ga_h))

        # instrumented pass: CUDA events around the three kernels of the neighbour step, then the model per batch
        V.event_log = {}
        try:
            sel = V.select_neighbors(structs, 4.0, 0.4, angle)
            batches = [sel.csr(s0, min(s0 + bs, S)) for s0 in range(0, S, bs)]
            torch.cuda.synchronize()
            ms = {k: sum(e0.elapsed_time(e1) for e0, e1 in v) for k, v in V.event_log.items()}
            passes = len(V.event_log.get("voronoi_neighbors", []))
        finally:
            V.event_log = None
        eng = model.engine
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for c in batches:                        # shapes are warm from the timed windows
            eng.predict_step(eng.load_batch_device_csr(c, *shape_class(c["M"], c["N"]), plan=False), replan=True)
        e0.record()
        for c in batches:
            eng.predict_step(eng.load_batch_device_csr(c, *shape_class(c["M"], c["N"]), plan=False), replan=True)
        e1.record()
        torch.cuda.synchronize()
        ms["model"] = e0.elapsed_time(e1)
        us = {k: 1e3 * v / S for k, v in ms.items()}
        host_rate, dev_rate = reps_h * S / t_h, reps_d * S / t_d
        lines.append(
            f"{name}: {S} structures, {atoms} atoms, {cfg_name} config (L{model.spec.n_attention}), batch {bs}; "
            f"host route {host_rate:,.0f} structures/s ({reps_h} passes in {t_h:.2f} s); predict_structures "
            f"{dev_rate:,.0f} structures/s ({reps_d} passes in {t_d:.2f} s), {dev_rate / host_rate:.1f}x; "
            f"CUDA events per structure: scann_voronoi_neighbors {us.get('voronoi_neighbors', 0):.2f} us "
            f"({passes} passes), scann_voronoi_select {us.get('voronoi_select', 0):.3f} us, scann_voronoi_batch_csr "
            f"{us.get('voronoi_batch_csr', 0):.3f} us, model (pack + plan + forward) {us['model']:.2f} us; "
            f"max |diff| y {dy:.1e}, ga {dga:.1e}")
        print(lines[-1], flush=True)
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
