"""Voronoi neighbour lists: GPU (scann_voronoi_neighbors via scann_b200.voronoi) against the scipy/Qhull oracle on the
same seeded structures -- QM9-like boxed molecules (9-29 atoms in a 20 Angstrom cube) and MP2018-like crystals (2-64
sites, triclinic).  Prints the card, the rates (structures/s, end to end from Python structures to the reference's
neighbour lists, device-synchronised, warmed up, window >= 1 s) and a parity summary.

    python tools/voronoi_bench.py [--n 2000] [--oracle-n 40] [--out voronoi_bench.log]
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import voronoi_oracle as VO                    # noqa: E402
from tests.test_voronoi import molecule, random_cell     # noqa: E402


def workloads(n, seed=0):
    rng = np.random.default_rng(seed)
    qm9 = [molecule(rng, int(rng.integers(9, 30))) for _ in range(n)]
    mp = [random_cell(rng, int(rng.integers(2, 65))) for _ in range(n)]
    return {"qm9_boxed": qm9, "mp2018_crystal": mp}


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                   # noqa: BLE001
        return f"unknown ({e})"


def rate(fn, min_s=1.0):
    fn()                                                     # warm-up (module load, first launches)
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
    ap.add_argument("--oracle-n", type=int, default=40)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    from scann_b200 import voronoi as V
    lines = [f"card: {card()}", f"torch {torch.__version__}, device {torch.cuda.get_device_name(0)}"]
    for name, structs in workloads(a.n).items():
        atoms = sum(len(s.cart_coords) for s in structs)
        reps, t = rate(lambda: V.compute_voronoi_neighbors(structs))      # ends in a stream synchronise
        gpu = reps * len(structs) / t
        sub = structs[:a.oracle_n]
        t0 = time.perf_counter()
        want = [VO.compute_voronoi_neighbor(s) for s in sub]
        cpu = len(sub) / (time.perf_counter() - t0)
        got = V.compute_voronoi_neighbors(sub)
        same = sum(all([(n[1], round(n[4], 9)) for n in g] == [(n[1], round(n[4], 9)) for n in w] for g, w in zip(gs, ws))
                   for gs, ws in zip(got, want))
        err = max((abs(x[2] - y[2]) / y[2] for gs, ws in zip(got, want) for g, w in zip(gs, ws) for x, y in zip(g, w)),
                  default=0.0)
        lines.append(f"{name}: {len(structs)} structures, {atoms} atoms; GPU {gpu:,.0f} structures/s "
                     f"({reps} passes in {t:.2f} s); CPU oracle (scipy Qhull, 1 core) {cpu:,.1f} structures/s on "
                     f"{len(sub)}; identical neighbour lists {same}/{len(sub)}, max rel solid-angle diff {err:.1e}")
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
