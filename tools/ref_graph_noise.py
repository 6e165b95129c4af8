"""Noise floor of the reference's OWN graph code at the full configurations of the GPU parity test
(tests/test_gpu_parity.py::FULL_CASES, same seeds): create_model of the reference executed on the functional
TensorFlow stand-in (tests/tf_shim.py) in fp32 and in fp64, beside the oracle restatement in the same two precisions.
CPU only, needs a checkout of the reference SCANN project.
usage: SCANN_REFERENCE_ROOT=<reference checkout> python tools/ref_graph_noise.py > profiles/<round>_reference_graph_noise.log"""
import os, sys, time, warnings
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
warnings.simplefilter("ignore")
import numpy as np, torch
from oracle import scann_oracle as O
from scann_b200.config import model_spec
from scann_b200.configs import get_config
from scann_b200.params import ParamLayout
from scann_b200.synth import make_batch
from tests.golden.make_golden import oracle_kwargs
from tests.ref_stubs import load_reference_graph
from tests.test_reference_graph import run_reference_graph, relerr

CASES = {"qm9_b128_l7": ("qm9", "qm9", 128, {}), "mp2018_b64_l9": ("mp2018", "mp2018", 64, {}),
         "fullerene_b128_l7": ("fullerene", "fullerene", 128, {}),
         "ptgp_b16_l11": ("ptgp", "ptgp", 16, {"g_update": False, "gaussian_d": 4.0})}
ref = load_reference_graph()
print("case | reference graph fp64 vs oracle fp64 (y, ga) | reference graph fp32 vs fp64 (y, ga) | oracle fp32 vs fp64 (y, ga) | "
      "largest per-tensor gradient error, reference graph fp32 vs fp64 (relative to the tensor's own maximum)")
for name, (cfg_name, shape, B, over) in CASES.items():
    t0 = time.time()
    cfg = get_config(cfg_name); cfg["model"].update(over)
    spec = model_spec(cfg); lay = ParamLayout(spec); w = lay.to_dict(lay.randomize_arena(21))
    ring = bool(spec.use_ring)
    inputs, target = make_batch(shape, 13, B=B, use_ring=ring)
    kw = dict(oracle_kwargs(spec), use_ring=ring)
    y64, ga64 = O.predict(w, inputs, torch.float64, **kw)
    y32, ga32 = O.predict(w, inputs, torch.float32, **kw)
    r64 = run_reference_graph(ref, cfg, w, inputs, target, dtype=torch.float64)
    r32 = run_reference_graph(ref, cfg, w, inputs, target, dtype=torch.float32)
    gerr = max((relerr(r32["grads"][k], r64["grads"][k]), k) for k in r64["grads"])
    print(f"{name} | {relerr(r64['y'], y64):.1e}, {relerr(r64['ga'], ga64):.1e} | {relerr(r32['y'], y64):.1e}, "
          f"{relerr(r32['ga'], ga64):.1e} | {relerr(y32, y64):.1e}, {relerr(ga32, ga64):.1e} | {gerr[0]:.1e} ({gerr[1]}) "
          f"| {time.time() - t0:.0f} s", flush=True)
