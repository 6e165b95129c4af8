#!/usr/bin/env python
"""Benchmark of the SCANN attention hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # our sm_100a path
    python bench.py --impl reference --gpus N --steps K ...   # reference restated on CPU
    python bench.py ... --dump-outputs DIR                    # + outputs of the last timed step as DIR/*.npy

Workload = BASELINE.json configs[1]: QM9 HOMO model (configs/model_qm9.yaml) train step
(forward + backward + Adam), 128 structures per GPU, synthetic QM9-shaped padded batch
(scann_b200/synth.py), random-init weights.  Weak scaling: every rank owns its own batch of 128;
one NCCL all-reduce of the gradient arena per step.

`value`   structures/s with the padded inputs already resident in HBM (plan + fwd + bwd + Adam).
`e2e`     same metric through the public API ``model.train_on_batch(numpy inputs, targets)``:
          host->device copies from pinned memory and a device->host read of the loss inside
          the timed region.
`roofline` the dominant kernel (local-attention backward) against measured HBM bandwidth.
`cpu_baseline` the oracle (PyTorch-CPU restatement of the reference graph; TensorFlow is not
          installable here) timed on the host cores for a bounded sample.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (config name in scann_b200.configs, synthetic shape, structures per GPU)
    "qm9": ("qm9", "qm9", 128),                 # BASELINE.json configs[1] (default, the headline)
    "mp2018": ("mp2018", "mp2018", 64),         # configs[2] / [4]: Materials Project shaped batches
    "fullerene": ("fullerene", "fullerene", 128),
    "ptgp": ("ptgp", "ptgp", 64),               # configs[3]: Pt/graphene MD model, 200-256 atoms, g_update=False, ring features
}

QM9_CONFIG = {
    "model": {"n_atoms": 10, "embedding_dim": 48, "n_attention": 7, "local_dim": 128, "num_head": 8,
              "global_dim": 128, "dense_out": 128, "scale": 0.5, "use_attn_norm": True, "use_ga_norm": True,
              "use_ring": False, "g_update": True, "gaussian_d": 4.0, "feature": "atomic", "use_drop": False},
    "hyper": {"batch_size": 128, "lr": 0.0005, "min_lr": 0.0001, "scheduler": "sgdr", "target": "homo"},
}
METRIC = "structures/sec (QM9 train step fwd+bwd+Adam, batch 128 per GPU)"


def workload_config(name):
    from scann_b200.configs import get_config
    if name == "qm9":
        return QM9_CONFIG, "qm9", 128, METRIC
    cfg_name, shape, B = WORKLOADS[name]
    cfg = get_config(cfg_name)
    if name == "ptgp":      # model_ptgp.yaml lacks these two keys (KeyError in the reference as shipped)
        cfg["model"].update(g_update=False, gaussian_d=4.0)
    cfg["hyper"].setdefault("lr", 1e-4)
    return cfg, shape, B, f"structures/sec ({name} train step fwd+bwd+Adam, batch {B} per GPU)"
UNIT = "structures/s"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


# --------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- CPU reference (oracle)
def cpu_train_step_fn():
    """One reference train step on the host: the oracle's fp32 restatement of the reference graph
    with reverse-mode autodiff + Keras Adam.  Returns (step_fn, cores)."""
    import torch
    from oracle import scann_oracle as O
    from scann_b200.config import model_spec
    from scann_b200.params import ParamLayout
    from scann_b200.synth import make_batch

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    spec = model_spec(QM9_CONFIG)
    lay = ParamLayout(spec)
    w = lay.to_dict(lay.init_arena(1))
    inp, tgt = make_batch("qm9", 0, B=128)
    l2n = [e.name for e in lay if e.l2]
    kw = dict(n_attention=spec.n_attention, g_update=True, gaussian_d=spec.gaussian_d, use_attn_norm=True,
              use_ga_norm=True)
    state = {"w": {k: v.copy() for k, v in w.items()}, "m": {k: np.zeros_like(v) for k, v in w.items()},
             "v": {k: np.zeros_like(v) for k, v in w.items()}, "t": 0}

    B_, M_ = inp["atomic"].shape
    gen = torch.Generator().manual_seed(0)

    def step():
        # training-mode Dropout(0.1) masks (scann_model.py:374, attention.py:29), as in a Keras fit step
        names = ["dense_embed"] + ["residual_norm" if l == 0 else f"residual_norm_{l}" for l in range(spec.n_attention)]
        masks = {n: (torch.rand(B_, M_, 128, generator=gen) >= 0.1).float() / 0.9 for n in names}
        _, _, _, g = O.loss_and_grads(state["w"], inp, tgt, l2n, dtype=torch.float32, drop_masks=masks, **kw)
        state["t"] += 1
        for k in state["w"]:
            state["w"][k], state["m"][k], state["v"][k] = O.adam_legacy_step(
                state["w"][k], g[k].astype(np.float32), state["m"][k], state["v"][k], state["t"], 5e-4)
        return 128

    step.workload = {"structures_per_gpu": 128, "M": int(M_), "N": int(inp["neighbors"].shape[2]),
                     "layers": int(spec.n_attention), "valid_atoms_per_gpu": int(inp["atom_mask"].sum()),
                     "valid_pairs_per_gpu": int(inp["neighbor_mask"].sum()), "dropout": 0.1}
    return step, cores


def emit(line: str) -> None:          # replaced in main(): stdout is reserved for this one line
    print(line)


def dump_outputs(out_dir, eng, b, batch_global):
    """Writes what the last timed train step computed, as float32 .npy files: ``loss`` = [loss, RMSE, MAE] (what
    ``model.train_on_batch`` returns), ``params`` = the parameter arena after its Adam update (``model.get_weights``
    in ParamLayout order), and ``y`` [B] / ``ga_score`` [B*M] of its training-mode forward (Dropout on).  The inputs,
    initial weights and Dropout seeds are fixed, so two builds can be compared file by file (about 3.6 MB for qm9).
    Expect two runs of one build to differ at float32 round-off, because atomic float32 sums are not ordered: of
    order 1e-5 of the largest magnitude in y and the loss, less in the parameters."""
    ws = eng._workspace(b, True)
    out = {"loss": eng.loss_value(batch_global)[:3], "params": eng.params, "y": ws["y"], "ga_score": ws["ga"]}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy().astype(np.float32))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    step, cores = cpu_train_step_fn()
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    n = 0
    for _ in range(args.steps):
        n += step()
    dt = time.perf_counter() - t0
    v = n / dt
    sample = f"{args.steps} train steps of one 128-structure QM9-shaped batch after {args.warmup} warm-up"
    emit(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the same seeded batch, model depth and Dropout sites as the sm_100a arm's N = 1 workload (same keys, same values)
        "config": dict({"workload": "qm9_train_step_b128"}, **step.workload,
                       note="reference graph restated on CPU in PyTorch (TensorFlow 2.10 is not installable in this "
                            "image; the restatement equals the reference's own create_model code run on a TensorFlow "
                            "stand-in, tests/test_reference_graph.py); rank 0 only"),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# --------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from scann_b200 import dist as sdist
    from scann_b200.model import create_model
    from scann_b200.synth import count_valid, make_batch

    rank, local_rank, world = sdist.init()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    CFG, shape_name, B, metric = workload_config(args.workload)
    model = create_model(CFG, seed=1)
    sdist.attach(model, world)
    eng = model.engine
    # the Keras train step runs the graph with training=True: Dropout(0.1) after dense_embed and in every
    # ResidualNorm is part of the measured step (the facade does the same in train_on_batch / fit)
    eng.train_dropout = True
    def rank_batch(shape, Bl, ring=False):
        """This rank's batch.  One GPU: the seeded batch of Bl structures.  N GPUs: the seeded GLOBAL batch of N * Bl
        structures, dealt to the ranks with equal structure counts and balanced pair counts (dist.balanced_shards:
        a data-parallel step is as slow as its slowest rank) -- per-GPU work stays what it is on one GPU."""
        if world == 1:
            return make_batch(shape, seed=rank, B=Bl, use_ring=ring)
        gin, gt = make_batch(shape, seed=0, B=Bl * world, use_ring=ring)
        mine = sdist.balanced_shards(gin["neighbor_mask"].reshape(Bl * world, -1).sum(1), world)[rank]
        return {k: np.ascontiguousarray(v[mine]) for k, v in gin.items()}, np.ascontiguousarray(gt[mine])

    inputs, target = rank_batch(shape_name, B, bool(CFG["model"].get("use_ring")))
    A_valid, P_valid = count_valid(inputs)
    lr = CFG["hyper"]["lr"]

    # device-resident copies of the padded inputs (the `value` arm starts from HBM)
    dev_inputs = {k: torch.from_numpy(np.ascontiguousarray(v.view(np.uint8) if v.dtype == np.bool_ else v)).to(dev)
                  for k, v in inputs.items()}
    tgt_dev = torch.from_numpy(target).to(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def step_device():
        b = eng.load_batch(dev_inputs, plan=False, pairs_hint=P_valid)   # device-to-device into the persistent buffers
        eng.train_step(b, tgt_dev, lr, allreduce=model.allreduce, batch_global=B * world, replan=True)
        return b

    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    eng.check_status()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- timed region 1: inputs resident in HBM
    launches0 = eng.launches
    evs = []
    barrier()
    for _ in range(args.steps):
        flush.fill_(1.0)                                   # L2 flush, outside the per-step events
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last_batch = step_device()
        e1.record()
        evs.append((e0, e1))
    barrier()
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    launches = eng.launches - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, last_batch, B * world)
    # ---- timed region 2: end to end through the public API (host buffers).  The call a user of the reference makes
    # is model.fit(iterator) (scann_model.py:232-241): every step packs the numpy batch into pinned memory, copies
    # it to the device (copy stream, overlapping the previous step), runs the step and reads [loss, rmse, mae] back
    # (asynchronous 16-byte copy per step, collected at the end of the epoch).
    class Repeat:
        """Sequence handing out the same host batch n times (len / __getitem__ like the reference's DataIterator)."""
        def __init__(self, item, n, ragged=False):
            self.item, self.n = item, n
            if ragged:
                self.csr_item = lambda i: self.item
        def __len__(self):
            return self.n
        def __getitem__(self, i):
            return self.item

    def timed_fit(item, ragged=False):
        model.fit(Repeat(item, 3, ragged), epochs=1, verbose=0)
        gc.collect()                     # a generation-2 collection inside a 20 ms wall-clock region is visible
        barrier()
        t0 = time.perf_counter()
        model.fit(Repeat(item, args.steps, ragged), epochs=1, verbose=0)
        barrier()
        return time.perf_counter() - t0, model.last_e2e_bytes

    e2e_s, (h2d, d2h) = timed_fit((inputs, target))
    # ---- 2a: the same through the blocking model.train_on_batch (loss returned to the caller every step)
    for _ in range(2):
        model.train_on_batch(inputs, target)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        model.train_on_batch(inputs, target)
    barrier()
    e2e_tob_s = time.perf_counter() - t0
    # ---- 2b: fit with the batch handed over in its ragged (CSR) form: only valid atoms / pairs travel and
    # scann_pack_batch pads on the device (scann_b200/datagenerator.py; extra line, not the headline)
    e2e_csr_s, h2d_csr = None, None
    try:
        from scann_b200.datagenerator import padded_to_csr
        e2e_csr_s, (h2d_csr, _) = timed_fit((padded_to_csr(inputs), target), ragged=True)
    except ValueError:
        pass
    clocks = sampler.stop() if rank == 0 else None
    # ---- instrumented pass: CUDA events around the local-attention kernels
    # (eager launches, one event pair per call: a ~2 ms spin kernel in front of every step lets the host enqueue the
    # whole step ahead of the GPU, so that an interval holds the kernels only and not the host's launch gaps)
    eng.prof = {}
    for _ in range(args.steps):
        flush.fill_(1.0)
        torch.cuda._sleep(4_000_000)
        step_device()
    torch.cuda.synchronize()
    prof = eng.prof_summary()
    eng.prof = None
    # ---- inference forward (reported beside the headline)
    for _ in range(3):
        eng.predict_step(eng.load_batch(dev_inputs, plan=False, pairs_hint=P_valid), replan=True)
    torch.cuda.synchronize()
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    i0.record()
    for _ in range(args.steps):
        eng.predict_step(eng.load_batch(dev_inputs, plan=False, pairs_hint=P_valid), replan=True)
    i1.record()
    torch.cuda.synchronize()
    infer_ms = i0.elapsed_time(i1)

    # ---- MP2018-shaped sub-record (BASELINE.json configs[4]: the data-parallel scaling sweep is quoted on
    # MP2018-shaped batches): the same two timed regions on model_mp2018.yaml, 64 structures per GPU
    mp_dev_ms = mp_e2e_ms = 0.0
    mp_info = None
    if args.workload == "qm9" and not args.no_mp2018:
        mcfg, mshape, mB, _ = workload_config("mp2018")
        mmodel = create_model(mcfg, seed=1)
        sdist.attach(mmodel, world)
        meng = mmodel.engine
        meng.train_dropout = True
        minputs, mtarget = rank_batch(mshape, mB)
        mA, mP = count_valid(minputs)
        mdev = {k: torch.from_numpy(np.ascontiguousarray(v.view(np.uint8) if v.dtype == np.bool_ else v)).to(dev)
                for k, v in minputs.items()}
        mtgt = torch.from_numpy(mtarget).to(dev)

        def mstep():
            bb = meng.load_batch(mdev, plan=False, pairs_hint=mP)
            meng.train_step(bb, mtgt, mcfg["hyper"]["lr"], allreduce=mmodel.allreduce, batch_global=mB * world, replan=True)

        for _ in range(max(args.warmup, 3)):
            mstep()
        barrier()
        mevs = []
        for _ in range(args.steps):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            mstep()
            e1.record()
            mevs.append((e0, e1))
        barrier()
        mp_dev_ms = sum(a.elapsed_time(b) for a, b in mevs)
        for _ in range(2):               # (the first fit of a model also allocates its staging buffers and streams)
            mmodel.fit(Repeat((minputs, mtarget), 3), epochs=1, verbose=0)
        gc.collect()
        barrier()
        t0 = time.perf_counter()
        mmodel.fit(Repeat((minputs, mtarget), args.steps), epochs=1, verbose=0)
        barrier()
        mp_e2e_ms = (time.perf_counter() - t0) * 1e3
        meng.check_status()
        mp_info = {"B": mB, "A": mA, "P": mP, "layers": mcfg["model"]["n_attention"], "h2d": mmodel.last_e2e_bytes[0]}

    t = torch.tensor([dev_ms, e2e_s * 1e3, infer_ms, (e2e_csr_s or 0.0) * 1e3, e2e_tob_s * 1e3, mp_dev_ms, mp_e2e_ms],
                     dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, infer_ms, e2e_csr_ms, e2e_tob_ms, mp_dev_ms, mp_e2e_ms = (float(x) for x in t.cpu())

    def finish():
        # Captured CUDA graphs hold NCCL work; tearing the communicator down under them can hang at
        # interpreter exit, so every rank synchronises, meets at a barrier and leaves without destructors.
        sys.stdout.flush()
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()
            os._exit(0)

    if rank != 0:
        finish()
        return

    L = CFG["model"]["n_attention"]
    peaks, peak_kind = measured_peaks()
    # algorithmic bytes per launch (DESIGN.md section 5): valid pairs P and atoms A only
    bytes_bwd = 1540.0 * P_valid + 1028.0 * A_valid
    bytes_fwd = 1028.0 * P_valid + 1028.0 * A_valid
    if not bool(CFG["model"].get("g_update", True)):
        # g_update = False (attention.py:155): no per-pair geometry tensor exists algorithmically -- a pair is its distance,
        # weight, neighbour index and mask (16 bytes, BASELINE.md section 3: 21 MB per layer on the full PtGP shape); the
        # per-atom rows are x, q, out forward and d_ctx, dq, dx backward.  This implementation materialises g' (512 bytes
        # per pair written and read back), so its fraction of THIS roofline is small by construction: the layer is bound
        # by the 3xTF32 key projection (550 flop per byte), see tensor_view.
        bytes_fwd = 16.0 * P_valid + 1028.0 * A_valid
        bytes_bwd = 16.0 * P_valid + 1540.0 * A_valid
    n_bwd, ms_bwd = prof.get("la_backward", (0, float("nan")))
    n_fwd, ms_fwd = prof.get("la_forward", (0, float("nan")))
    n_wg, ms_wg = prof.get("wgrad_batch", (0, float("nan")))
    ach = bytes_bwd / (ms_bwd * 1e-3) / 1e9
    pipe_bwd = eng.tc_la_bwd and (eng.la_pipe & 12) == 12 and int(inputs["neighbors"].shape[2]) <= 32 and \
        bool(CFG["model"].get("g_update", True))
    noup_pipe = eng.tc_la_bwd and getattr(eng, "noup_pipe", False) and int(inputs["neighbors"].shape[2]) <= 32 and \
        not bool(CFG["model"].get("g_update", True))
    kern = ("la_attn_bwd_pipe_kernel + la_geom_bwd_pipe_kernel (one layer of local-attention backward: warp-specialised "
            "TMA pipelines, la_pipe_bwd.cu)" if pipe_bwd else
            "la_attn_bwd_pipe_kernel + noupdate_geom_bwd_kernel (one layer of local-attention backward of a g_update = "
            "False model: pipelined attention kernel, la_pipe_bwd.cu, + filter gradient)" if noup_pipe else
            "la_attn_bwd_tc_kernel + la_geom_bwd_tc_kernel (one scann_la_backward_tc call = one layer of "
            "local-attention backward)" if eng.tc_la_bwd else "la_bwd_simt_kernel")
    # DRAM traffic of the same kernels from the committed `ncu --set full` capture (dram__bytes_read.sum +
    # dram__bytes_write.sum per launch), when the workload matches the capture
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        if tj.get("workload") == f"{args.workload}_train_step_b{B}":
            traffic = tj.get("la_backward_bytes_per_launch")
    # tensor-core view of the same kernels: 3xTF32 = 3 tensor-core products per algorithmic product
    # (two [P,128]x[128,128] input-gradient GEMMs per layer = 65 536 flops per valid pair; the weight
    # gradients are a separate launch)
    flops_bwd = 3.0 * (65536.0 if bool(CFG["model"].get("g_update", True)) else 32768.0) * P_valid    # one GEMM without geometry update
    roof = {"bound": "hbm", "kernel": kern, "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": ach / peaks["hbm_gbs"], "traffic": traffic, "peak_kind": peak_kind,
            "launches_timed": n_bwd, "ms_per_launch": ms_bwd,
            "share_of_step": n_bwd * ms_bwd / args.steps / (dev_ms / args.steps),
            "algorithmic_bytes_per_launch": bytes_bwd,
            # measured kind::tf32 rate of one SM (profiles/r02_tf32_peak.md: 64.5 cycles per 128x128x8 tcgen05.mma, the math
            # floor of the N = 128 form = 4 064 flop/clk/SM), times the SMs and the SM clock seen during this run
            "tensor_view": (lambda tf, pk: {"tf32_tflops_issued": tf, "tf32_peak_measured_tflops": pk, "frac": tf / pk,
                                            "note": "3 tf32 products per fp32 product; peak = 4064 flop/clk/SM (measured "
                                                    "tcgen05 kind::tf32 rate, M = N = 128) x SMs x SM clock"})(
                flops_bwd / (ms_bwd * 1e-3) / 1e12,
                4064.0 * eng.sm_count * ((clocks or {}).get("sm_mhz") or 1965.0) * 1e6 / 1e12),
            "la_forward": {"achieved": bytes_fwd / (ms_fwd * 1e-3) / 1e9, "ms_per_launch": ms_fwd,
                           "frac": bytes_fwd / (ms_fwd * 1e-3) / 1e9 / peaks["hbm_gbs"]}}
    if n_wg:
        # every weight-gradient GEMM of the step in one launch: reads each saved per-pair tensor once
        # (per pair and layer: g', d_k, g, d_pre + the gathered x[j]; per atom: x, s_pre, t, dq and the four
        # ResidualNorm operands -- models without geometry update have no g / d_pre / s_pre / t problems)
        # (the gathered neighbour rows x[j] of the key-kernel problem come out of the [A,128] atom array, which stays in
        # L2: they are counted once per atom, not once per pair)
        gu = bool(CFG["model"].get("g_update", True))
        bytes_wg = L * ((4 if gu else 2) * 512.0 * P_valid + (9 if gu else 7) * 512.0 * A_valid)
        roof["wgrad_batch"] = {"achieved": bytes_wg / (ms_wg * 1e-3) / 1e9, "ms_per_launch": ms_wg,
                               "frac": bytes_wg / (ms_wg * 1e-3) / 1e9 / peaks["hbm_gbs"]}
    # global attention + head (one CTA per structure): algorithmic bytes 516 A + 512 B forward (q|k rows in, ga out,
    # pooled context), twice that backward; a few microseconds of launch-latency-bound work per step
    n_gaf, ms_gaf = prof.get("ga_forward", (0, float("nan")))
    n_gab, ms_gab = prof.get("ga_backward", (0, float("nan")))
    if n_gaf:
        bytes_ga = 2 * 516.0 * A_valid + 512.0 * B
        roof["global_attention"] = {
            "kernel": ("ga_head_fwd_staged_kernel / ga_head_bwd_staged_kernel (GlobalAttention + property head, one CTA per "
                       "structure, its query | key block staged in shared memory; ga.cu)"
                       if int(inputs["neighbors"].shape[1]) * 1024 + 8192 <= 200 * 1024 else
                       "ga_head_fwd_kernel / ga_head_bwd_kernel (GlobalAttention + property head, one CTA per structure; the "
                       "query | key block of a structure this large does not fit shared memory)"),
            "forward": {"achieved": bytes_ga / (ms_gaf * 1e-3) / 1e9, "ms_per_launch": ms_gaf,
                        "frac": bytes_ga / (ms_gaf * 1e-3) / 1e9 / peaks["hbm_gbs"], "algorithmic_bytes": bytes_ga},
            "backward": (None if not n_gab else
                         {"achieved": 2 * bytes_ga / (ms_gab * 1e-3) / 1e9, "ms_per_launch": ms_gab,
                          "frac": 2 * bytes_ga / (ms_gab * 1e-3) / 1e9 / peaks["hbm_gbs"]}),
            "note": "1-2 MB per launch: bound by launch latency and the per-structure reduction chain, not by HBM"}
    # bounded CPU sample (rank 0, N=1 only)
    cpu = None
    if world == 1 and not args.no_cpu and args.workload == "qm9":
        step, cores = cpu_train_step_fn()
        step()
        t0 = time.perf_counter()
        n = 0
        while time.perf_counter() - t0 < args.cpu_seconds:
            n += step()
        cpu = {"value": n / (time.perf_counter() - t0), "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{n // 128} train steps of the same 128-structure batch (~{args.cpu_seconds:.0f} s), "
                         "PyTorch-CPU restatement of the reference graph (TensorFlow not installable)"}
    out = {
        "metric": metric, "value": B * world * args.steps / (dev_ms * 1e-3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}_train_step_b{B}", "structures_per_gpu": B,
                   "M": int(inputs["neighbors"].shape[1]), "N": int(inputs["neighbors"].shape[2]), "layers": L,
                   "valid_atoms_per_gpu": A_valid, "valid_pairs_per_gpu": P_valid, "parallelism": f"dp{world}",
                   "sharding": ("one seeded batch" if world == 1 else
                                "seeded global batch dealt to the ranks: equal structure counts, balanced pair counts"),
                   "l2": "flushed between steps (256 MiB write outside the timed events)",
                   "engine": "tcgen05 3xTF32 (fp32-accurate)" if eng.tc_la_bwd else "fp32 SIMT",
                   "dropout": eng.dropout_rate if eng.train_dropout else 0.0,
                   "cuda_graphs": bool(eng.use_graphs)},
        "e2e": {"value": B * world * args.steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h),
                "api": "model.fit(Sequence of host numpy batches): per step one pinned blob -> device copy on a copy "
                       "stream + one 16-byte loss read-back, losses collected at the end of the epoch"},
        "e2e_train_on_batch": {"value": B * world * args.steps / (e2e_tob_ms * 1e-3), "unit": UNIT,
                               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                               "note": "blocking model.train_on_batch: the loss is returned to the caller every step"},
        "e2e_ragged_input": (None if not e2e_csr_ms else
                             {"value": B * world * args.steps / (e2e_csr_ms * 1e-3), "unit": UNIT,
                              "h2d_bytes_per_step": int(h2d_csr), "d2h_bytes_per_step": 16,
                              "note": "fit over CSR batches: valid atoms / pairs only, padded on the device"}),
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roof,
        "cpu_baseline": cpu,
        "infer": {"value": B * world * args.steps / (infer_ms * 1e-3), "unit": UNIT,
                  "note": "forward incl. ga_score, inputs resident in HBM"},
        "mp2018": (None if mp_info is None else {
            "metric": f"structures/sec (mp2018 train step fwd+bwd+Adam, batch {mp_info['B']} per GPU)",
            "value": mp_info["B"] * world * args.steps / (mp_dev_ms * 1e-3), "unit": UNIT,
            "ms_per_step": mp_dev_ms / args.steps,
            "e2e": {"value": mp_info["B"] * world * args.steps / (mp_e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": int(mp_info["h2d"]), "d2h_bytes_per_step": 16},
            "config": {"workload": f"mp2018_train_step_b{mp_info['B']}", "layers": mp_info["layers"],
                       "valid_atoms_per_gpu": mp_info["A"], "valid_pairs_per_gpu": mp_info["P"], "parallelism": f"dp{world}"}}),
    }
    emit(json.dumps(out))
    finish()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the bounded CPU baseline sample")
    ap.add_argument("--no-mp2018", action="store_true", help="skip the MP2018-shaped sub-record")
    ap.add_argument("--workload", default="qm9", choices=sorted(WORKLOADS),
                    help="qm9 (default, BASELINE.json configs[1]) | mp2018 | fullerene: other shapes, for reference")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed train step computed to DIR/<name>.npy (sm_100a arm only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the sm_100a arm (--impl ours)")
    # stdout carries exactly ONE JSON line.  Libraries write there too (NCCL prints "NCCL version ..." to stdout
    # under NCCL_DEBUG=VERSION, whatever NCCL_DEBUG_FILE says), so file descriptor 1 points at stderr until the
    # line is printed.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    global emit

    def emit(line: str) -> None:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(line)
        sys.stdout.flush()
        os.dup2(2, 1)

    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
