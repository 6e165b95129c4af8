"""Train-step time of the default and the deterministic mode on the same GPU (DESIGN.md section 4.7).

For every workload two engines with the same parameters train on the same pre-loaded batches; the two are timed in
alternating windows of CUDA-event-timed graph replays, and the median window of each is reported.  Usage:
    python tools/det_time.py [--steps 50] [--windows 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from scann_b200.config import model_spec          # noqa: E402
from scann_b200.configs import get_config         # noqa: E402
from scann_b200.engine import Engine              # noqa: E402
from scann_b200.params import ParamLayout         # noqa: E402
from scann_b200.synth import make_batch           # noqa: E402

# name -> (config, batch shape, B, model overrides, training-mode Dropout)
WORKLOADS = {
    "qm9_b128_dropout": ("qm9", "qm9", 128, {}, True),
    "mp2018_b64": ("mp2018", "mp2018", 64, {}, False),
    "fullerene_b128": ("fullerene", "fullerene", 128, {}, False),
    "ptgp_b64": ("ptgp", "ptgp", 64, {"g_update": False, "gaussian_d": 4.0}, False),
}


def step_ms(eng, batches, steps):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(steps):
        b, y = batches[i % len(batches)]
        eng.train_step(b, y, lr=1e-4)
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def kernel_breakdown(engines, steps):
    """Device time per kernel name and step, default vs deterministic, for the kernels whose time differs (a separate,
    profiled run: tracing slows the host)."""
    from torch.profiler import ProfilerActivity, profile
    per = {}
    for det, (eng, batches) in engines.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step_ms(eng, batches, steps)
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            if t > 0:
                per.setdefault(ev.key[:60], [0.0, 0.0])[int(det)] += t / steps
    diff = {k: [round(a, 2), round(b, 2)] for k, (a, b) in per.items() if abs(a - b) >= 0.5}
    return dict(sorted(diff.items(), key=lambda kv: -abs(kv[1][1] - kv[1][0])))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--out", default="")
    ap.add_argument("--profile", type=int, default=10, help="steps per engine under torch.profiler (0: off)")
    args = ap.parse_args()
    dev = torch.cuda.get_device_properties(0)
    lines = [f"# device: {dev.name}, {dev.multi_processor_count} SMs"]
    try:
        import subprocess
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        lines.append("# power limit, max SM clock: " + q.stdout.strip())
    except Exception as e:         # noqa: BLE001 -- the query is informational
        lines.append(f"# nvidia-smi query failed: {e}")
    for name, (cfg_name, shape, B, over, drop) in WORKLOADS.items():
        cfg = get_config(cfg_name)
        cfg["model"].update(over)
        spec = model_spec(cfg)
        arena = ParamLayout(spec).randomize_arena(1)
        ring = bool(spec.use_ring)
        data = [make_batch(shape, 100 + i, B=B, use_ring=ring) for i in range(4)]
        res = {"workload": name}
        engines = {}
        for det in (False, True):
            eng = Engine(spec, arena, deterministic=det)
            eng.train_dropout = drop
            batches = []
            for inputs, target in data:
                b = eng.load_batch(inputs)
                batches.append((b, torch.from_numpy(target).cuda()))
            try:
                step_ms(eng, batches, 4)                         # capture + warm-up
            except NotImplementedError as e:
                res["det_refused"] = str(e)
                break
            n0 = eng.launches
            step_ms(eng, batches, 1)
            res["launches_" + ("det" if det else "default")] = eng.launches - n0
            engines[det] = (eng, batches)
        times = {False: [], True: []}
        for _ in range(args.windows):
            for det, (eng, batches) in engines.items():
                times[det].append(step_ms(eng, batches, args.steps))
        res["default_ms"] = round(float(np.median(times[False])), 4)
        if True in engines:
            res["det_ms"] = round(float(np.median(times[True])), 4)
            res["ratio"] = round(res["det_ms"] / res["default_ms"], 4)
            if args.profile:
                res["kernel_us_per_step"] = kernel_breakdown(engines, args.profile)
        res["windows_ms"] = {"default": [round(t, 4) for t in times[False]], "det": [round(t, 4) for t in times[True]]}
        lines.append(json.dumps(res))
        print(lines[-1], flush=True)
        engines.clear()
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
