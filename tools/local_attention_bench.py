"""What the local-attention scores cost: ``predict_structures`` and ``predict`` with and without
``local_attention=True`` on one GPU.

Workloads: QM9-like boxed molecules under the QM9 config (7 layers, batch 128) and MP2018-like crystals under the MP2018
config (9 layers, batch 64), the generators of tools/voronoi_bench.py, seeded weights; ``predict`` runs on one synthetic
host batch of the same config (scann_b200.synth, QM9 128 x 29 x 16 / MP2018 64 x 64 x 24).  Reports
- structures/s of predict_structures without and with the scores;
- structures/s of predict on the host batch without and with the scores;
- CUDA-event time of one unpack launch (scann_attn_to_csr for the structures route, scann_attn_to_padded for predict),
  mean over the batches of one instrumented pass outside the timed windows;
- bytes copied back to the host per structure for the scores (and, for predict_structures, the pair lists).
Every shape is warmed up first; timed windows are >= 1 s and end in a device synchronise, and the runs with and without
scores alternate (three rounds, the best of each is reported).

    python tools/local_attention_bench.py [--n 2000] [--out profiles/r03_local_attention.log]
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

CONFIGS = {"qm9_boxed": ("qm9", "qm9", 128), "mp2018_crystal": ("mp2018", "mp2018", 64)}


def rate(fn, min_s=1.0):
    """Calls per second of ``fn`` (which ends in a device synchronise) over a window of at least min_s."""
    reps, t = 0, 0.0
    t0 = time.perf_counter()
    while t < min_s:
        fn()
        reps += 1
        t = time.perf_counter() - t0
    return reps / t


def best_of_alternating(fns, rounds=3):
    best = [0.0] * len(fns)
    for fn in fns:
        fn()                                    # warm-up: every shape class, both graphs
    for _ in range(rounds):
        for i, fn in enumerate(fns):
            best[i] = max(best[i], rate(fn))
    return best


def unpack_ms(eng, steps):
    """Mean CUDA-event time of the unpack launch over ``steps()`` (eager forward, events around each launch)."""
    import torch
    eng.prof = {}
    try:
        steps()
        torch.cuda.synchronize()
        n, ms = eng.prof_summary()["attn_unpack"]
    finally:
        eng.prof = None
    return n, ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=2000)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    from scann_b200.config import model_spec
    from scann_b200.configs import get_config
    from scann_b200.model import create_model, shape_class
    from scann_b200.params import ParamLayout
    from scann_b200.synth import make_batch
    from scann_b200 import voronoi as V

    lines = [f"card: {card()}", f"torch {torch.__version__}, device {torch.cuda.get_device_name(0)}"]
    for name, structs in workloads(a.n).items():
        cfg_name, shape, bs = CONFIGS[name]
        cfg = get_config(cfg_name)
        model = create_model(cfg, infer=True, arena=ParamLayout(model_spec(cfg)).randomize_arena(3))
        eng = model.engine
        L = model.spec.n_attention
        S = len(structs)
        inputs, _ = make_batch(shape, 5, B=bs)
        B = inputs["atomic"].shape[0]

        def structures(la):
            return lambda: model.predict_structures(structs, batch_size=bs, local_attention=la)

        def host_batch(la):
            return lambda: model.predict(inputs, local_attention=la)

        s_off, s_on, p_off, p_on = best_of_alternating([structures(False), structures(True), host_batch(False),
                                                        host_batch(True)])
        # outputs: the flag changes neither y nor ga; bytes of the scores (and pair lists) that reach the host
        y0, ga0 = model.predict_structures(structs, batch_size=bs)
        y1, ga1, la = model.predict_structures(structs, batch_size=bs, local_attention=True)
        same_s = np.array_equal(y0, y1) and all(np.array_equal(g, h) for g, h in zip(ga0, ga1))
        pairs = sum(t.scores.shape[2] for t in la)
        s_bytes = sum(t.site_offsets.nbytes + t.neighbors.nbytes + t.distances.nbytes + t.scores.nbytes for t in la)
        model.predict(inputs)
        base_bytes = model.last_e2e_bytes[1]
        out_p = model.predict(inputs, local_attention=True)
        p_bytes = model.last_e2e_bytes[1] - base_bytes
        same_p = all(np.array_equal(g, h) for g, h in zip(model.predict(inputs), out_p[:2]))

        # instrumented pass: one unpack launch per batch, CUDA events around it
        sel = V.select_neighbors(structs, 4.0, 0.4, bool(model.spec.g_update))
        batches = [sel.csr(s0, min(s0 + bs, S)) for s0 in range(0, S, bs)]

        def csr_steps():
            for c in batches:
                b = eng.load_batch_device_csr(c, *shape_class(c["M"], c["N"]), plan=False)
                eng.predict_step(b, replan=True, local_attention="csr")

        n_csr, ms_csr = unpack_ms(eng, csr_steps)
        n_pad, ms_pad = unpack_ms(eng, lambda: [model.predict(inputs, local_attention=True) for _ in range(20)])
        lines.append(
            f"{name}: {S} structures, {pairs} kept pairs, {cfg_name} config (L{L}), batch {bs}; "
            f"predict_structures {s_off * S:,.0f} -> {s_on * S:,.0f} structures/s with local_attention ({s_on / s_off:.3f}x); "
            f"scann_attn_to_csr {1e3 * ms_csr:.1f} us per batch ({n_csr} launches), {1e3 * ms_csr * len(batches) / S:.3f} "
            f"us per structure; copied back for the scores {s_bytes / S:,.0f} B per structure "
            f"(L*8*4 = {L * 32} B per pair + offsets, neighbours, distances); y / ga unchanged: {same_s}")
        lines.append(
            f"{name} host batch {B} x {inputs['neighbors'].shape[1]} x {inputs['neighbors'].shape[2]}: predict "
            f"{p_off * B:,.0f} -> {p_on * B:,.0f} structures/s with local_attention ({p_on / p_off:.3f}x); "
            f"scann_attn_to_padded {1e3 * ms_pad:.1f} us per batch ({n_pad} launches); copied back for the scores "
            f"{p_bytes / B:,.0f} B per structure ([L, 8, M, N] fp32); y / ga unchanged: {same_p}")
        print(lines[-2], lines[-1], sep="\n", flush=True)
        eng.check_status()
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
