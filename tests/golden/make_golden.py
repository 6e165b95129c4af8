"""Generates tests/golden/*.npz from the fp64 oracle (oracle/scann_oracle.py).

TensorFlow is absent (SURVEY.md F2) and the reference ships no golden vectors (F8).  The fixtures are written by
the oracle; ``tests/test_reference_graph.py::test_golden_vectors_equal_the_reference_graph`` then runs the
reference's OWN ``create_model`` graph (imported from the SCANN_REFERENCE_ROOT checkout on the functional TensorFlow stand-in
``tests/tf_shim.py``) on the same seeded cases and requires equality at fp64 round-off, so the committed values are
pinned to reference-run code at the graph level (TensorFlow's own primitive kernels stay unpinned).

    python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import scann_oracle as O          # noqa: E402
from scann_b200.config import model_spec      # noqa: E402
from scann_b200.configs import get_config     # noqa: E402
from scann_b200.params import ParamLayout     # noqa: E402
from scann_b200.synth import make_batch       # noqa: E402

CASES = {
    # name: (config, shape, B, n_attention override, param seed, batch seed)
    "qm9_b4": ("qm9", "qm9", 4, None, 2, 10),
    "mp2018_b3_l3": ("mp2018", "mp2018", 3, 3, 3, 11),
    "fullerene_b2_l2": ("fullerene", "fullerene", 2, 2, 4, 12),
}


def oracle_kwargs(spec):
    return dict(n_attention=spec.n_attention, g_update=spec.g_update, gaussian_d=spec.gaussian_d,
                use_attn_norm=spec.use_attn_norm, use_ga_norm=spec.use_ga_norm)


def build_case(name):
    cfg_name, shape, B, L, pseed, bseed = CASES[name]
    cfg = get_config(cfg_name)
    if L is not None:
        cfg["model"]["n_attention"] = L
    spec = model_spec(cfg)
    lay = ParamLayout(spec)
    arena = lay.randomize_arena(pseed)
    inputs, target = make_batch(shape, bseed, B=B)
    return cfg, spec, lay, arena, inputs, target


def main():
    for name in CASES:
        cfg, spec, lay, arena, inputs, target = build_case(name)
        w = lay.to_dict(arena)
        l2n = [e.name for e in lay if e.l2]
        loss, y, ga, grads = O.loss_and_grads(w, inputs, target, l2n, dtype=torch.float64, **oracle_kwargs(spec))
        garena = lay.from_dict({k: v.astype(np.float32) for k, v in grads.items()})
        # grads kept as float64 per-tensor max / checksum plus a float32 arena (small models: < 5 MB -> store
        # only a strided sample to keep the fixture small)
        idx = np.arange(0, lay.total, 97)
        np.savez_compressed(os.path.join(HERE, f"{name}.npz"), y=y, ga=ga, loss=np.float64(loss),
                            grad_sample=garena[idx].astype(np.float64), grad_idx=idx,
                            grad_l2norm=np.float64(np.sqrt(sum((g.astype(np.float64) ** 2).sum() for g in grads.values()))))
        print(name, "loss", loss, "y", y.ravel()[:3])


if __name__ == "__main__":
    main()
