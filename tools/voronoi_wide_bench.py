"""Slabs with vacuum through the structure routes: the wide form of the Voronoi cell search (cells of up to 256 facets).

For 512 PtGP-like slab structures (a graphene sheet with a Pt cluster of 4-13 atoms) at each cell height c = 10, 15,
20 and 25 Angstrom: the structures the routes refuse (a cell beyond the capacity), the rates of
``compute_voronoi_neighbors`` and of ``predict_structures`` (PtGP config with ring flags, batch 64), the number of sites
that run the wide form and the CUDA-event time per centre of the narrow and the wide cell search.  With
``--parent-lib``, ``tools/voronoi_bench.py`` (QM9-like boxed molecules, MP2018-like crystals) runs alternately on that
library and on this tree's, to show that the narrow route kept its speed.  Card name and power limit are read in the
same call.

    python tools/voronoi_wide_bench.py [--n 512] [--parent-lib PATH] [--out profiles/r03_voronoi_wide.log]
"""
from __future__ import annotations

import argparse
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.voronoi_bench import card, rate                                    # noqa: E402
from tests.test_ring_routes import PTGP, _ring_model                          # noqa: E402
from tests.test_voronoi_wide import flags_of, slab                            # noqa: E402


def slab_set(n, c, seed=0):
    rng = np.random.default_rng(seed)
    return [slab(rng, c, int(rng.integers(4, 14))) for _ in range(n)]


def dropped(V, structs):
    """Structures whose neighbour lists raise (a cell beyond the capacity), counted one by one only if the set raises."""
    try:
        V.compute_voronoi_neighbors(structs)
        return []
    except ValueError:
        bad = []
        for k, s in enumerate(structs):
            try:
                V.compute_voronoi_neighbors([s])
            except ValueError:
                bad.append(k)
        return bad


def pass_times(V, structs):
    """One select_neighbors: per form (narrow / wide) the centres launched and the CUDA-event time of the cell search."""
    import torch
    sizes = {}
    run = V._select_pass

    def counted(*a, **k):
        cap = k.get("cap", a[11] if len(a) > 11 else V._CAP)
        sizes.setdefault(cap > V._CAP, []).append(len(a[4]))
        return run(*a, **k)
    V._select_pass, V.event_log = counted, {}
    try:
        V.select_neighbors(structs)
        torch.cuda.synchronize()
        log = V.event_log
    finally:
        V._select_pass, V.event_log = run, None
    out = {}
    for wide, name in ((False, "voronoi_neighbors"), (True, "voronoi_neighbors_wide")):
        ms = sum(e0.elapsed_time(e1) for e0, e1 in log.get(name, []))
        out[wide] = (sum(sizes.get(wide, [])), len(log.get(name, [])), ms)
    return out


def narrow_rates(lib, n):
    env = dict(os.environ)
    if lib:
        env["SCANN_B200_LIB"] = lib
    else:
        env.pop("SCANN_B200_LIB", None)
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "voronoi_bench.py"), "--n", str(n),
                          "--oracle-n", "4"], capture_output=True, text=True, env=env, timeout=1800)
    if res.returncode != 0:
        raise RuntimeError(res.stdout + res.stderr)
    return {m.group(1): float(m.group(2).replace(",", ""))
            for m in re.finditer(r"^(\w+): .*?GPU ([\d,]+) structures/s", res.stdout, re.M)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--heights", default="10,15,20,25")
    ap.add_argument("--parent-lib", default="")
    ap.add_argument("--narrow-n", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    from scann_b200 import voronoi as V
    lines = [f"card: {card()}", f"torch {torch.__version__}, device {torch.cuda.get_device_name(0)}"]
    model, _ = _ring_model("ptgp", **PTGP)
    for c in (float(h) for h in a.heights.split(",")):
        structs = slab_set(a.n, c)
        atoms = sum(len(s.atomic_numbers) for s in structs)
        bad = dropped(V, structs)
        keep = [s for k, s in enumerate(structs) if k not in set(bad)]
        flags = flags_of(keep)
        reps, t = rate(lambda: V.compute_voronoi_neighbors(keep))
        r_lists = reps * len(keep) / t
        out = model.predict_structures(keep, batch_size=64, ring_aromatic=flags)            # warm-up of the classes
        reps2, t2 = rate(lambda: model.predict_structures(keep, batch_size=64, ring_aromatic=flags))
        r_pred = reps2 * len(keep) / t2
        pt = pass_times(V, keep)
        (cn, ln, msn), (cw, lw, msw) = pt[False], pt[True]
        lines.append(
            f"c = {c:.0f} A: {len(structs)} structures, {atoms} atoms, dropped {len(bad)}; compute_voronoi_neighbors "
            f"{r_lists:,.0f} structures/s ({reps} passes in {t:.2f} s); predict_structures (ptgp L11, ring flags, "
            f"batch 64) {r_pred:,.0f} structures/s ({reps2} passes in {t2:.2f} s); select_neighbors: narrow "
            f"{cn} centres in {ln} launches, {msn:.2f} ms, {1e3 * msn / max(cn, 1):.2f} us/centre; wide {cw} centres "
            f"in {lw} launches, {msw:.2f} ms, {1e3 * msw / max(cw, 1):.2f} us/centre")
        print(lines[-1], flush=True)
        assert np.isfinite(out[0]).all()
    if a.parent_lib:
        runs = {"parent": [], "this": []}
        for r in range(a.reps):
            for name, lib in (("parent", a.parent_lib), ("this", "")):
                runs[name].append(narrow_rates(lib, a.narrow_n))
        for w in ("qm9_boxed", "mp2018_crystal"):
            p = [x[w] for x in runs["parent"]]
            n = [x[w] for x in runs["this"]]
            lines.append(f"voronoi_bench {w} ({a.narrow_n} structures), alternating runs: parent "
                         f"{', '.join(f'{v:,.0f}' for v in p)} structures/s; this tree "
                         f"{', '.join(f'{v:,.0f}' for v in n)} structures/s; medians {np.median(p):,.0f} / "
                         f"{np.median(n):,.0f} ({100 * (np.median(n) / np.median(p) - 1):+.1f} %), spread of the "
                         f"parent {100 * (max(p) - min(p)) / np.median(p):.1f} %")
            print(lines[-1], flush=True)
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
