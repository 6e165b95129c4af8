"""Voronoi neighbour lists on the GPU: the reference's ``compute_voronoi_neighbor`` (scann/utils/voronoi_neighbor.py:11-61)
without pymatgen.

The reference calls pymatgen's ``VoronoiNN(weight="solid_angle").get_voronoi_polyhedra`` per site (one Qhull
tessellation of every periodic image within ``cutoff``) and keeps the facets within ``d_thresh`` whose solid angle,
normalised by the site's largest, is at least ``w_thresh``.  Here every site of every structure is one warp of
``scann_voronoi_neighbors`` (csrc/voronoi.cu, fp64); pymatgen's retry loop -- a site whose cell still has an unbounded
facet is run again with ``cutoff = min(2 cutoff, longest cell diagonal + 0.011)`` -- re-launches only those sites.

A structure is anything with ``.cart_coords`` ``[n, 3]`` and ``.lattice.matrix`` ``[3, 3]`` (rows = lattice vectors),
e.g. a pymatgen ``Structure``.  A molecule must be boxed first (pymatgen: ``Molecule.get_boxed_structure``).
"""
from __future__ import annotations

import ctypes
from typing import List, Sequence

import numpy as np
import torch

from scann_b200 import _abi

ERR_COINCIDENT, ERR_CAPACITY, ERR_NO_FACET, ERR_TOPOLOGY = 32, 64, 128, 256
_INFINITE = 1
_CAP = 64                       # facet records per centre (the kernel's facet capacity)
_CHUNK = 1 << 16                # centres per launch
FACET = np.dtype([("solid_angle", "<f8"), ("normalized", "<f8"), ("distance", "<f8"), ("site", "<i4"),
                  ("image", "<i4")])
_MESSAGES = {ERR_COINCIDENT: "two points of its Voronoi point set are closer than 1e-8 Angstrom",
             ERR_CAPACITY: "its Voronoi cell exceeds the kernel's capacity (64 facets, 32 vertices per facet, 128 "
                           "points in one distance shell, images up to 511 cells away)",
             ERR_NO_FACET: "its Voronoi cell has no finite facet",
             ERR_TOPOLOGY: "a cut of its Voronoi cell was numerically inconsistent"}


def max_cutoff(lattice) -> float:
    """pymatgen's cap of the retry loop: the longest of the four cell diagonals, plus 0.01."""
    corners = np.array([[1, 1, 1], [-1, 1, 1], [1, -1, 1], [1, 1, -1]], np.float64)
    return float(np.linalg.norm(corners @ np.asarray(lattice, np.float64), axis=1).max()) + 0.01


def _arrays(structs):
    lats, xs = [], []
    for k, st in enumerate(structs):
        lat = getattr(st, "lattice", None)
        if lat is None:
            raise ValueError(f"structure {k} has no lattice: the Voronoi search is periodic, box a molecule first "
                             "(pymatgen: Molecule.get_boxed_structure)")
        L = np.asarray(lat.matrix, np.float64).reshape(3, 3)
        if not abs(np.linalg.det(L)) > 0:
            raise ValueError(f"structure {k}: singular lattice")
        X = np.asarray(st.cart_coords, np.float64).reshape(-1, 3)
        if not np.isfinite(X).all() or not np.isfinite(L).all():
            raise ValueError(f"structure {k}: non-finite coordinates")
        lats.append(L)
        xs.append(X)
    return lats, xs


def _run(lat, X, sa_off, atoms, cut, allow_pathological):
    """One launch over the listed centres -> (off [C+1], flags [C], records)."""
    _abi.require_gpu()
    dev = torch.device("cuda", torch.cuda.current_device())
    C = len(atoms)
    cs = np.searchsorted(sa_off, atoms, side="right") - 1
    d_lat = torch.from_numpy(lat).to(dev)
    d_x = torch.from_numpy(X).to(dev)
    d_sa = torch.from_numpy(sa_off.astype(np.int32)).to(dev)
    d_at = torch.from_numpy(atoms.astype(np.int32)).to(dev)
    d_cs = torch.from_numpy(cs.astype(np.int32)).to(dev)
    d_cut = torch.from_numpy(np.ascontiguousarray(cut, np.float64)).to(dev)
    head = (4 * (2 * C + 1) + 31) // 32 * 32
    nbytes = head + FACET.itemsize * C * _CAP
    slots = torch.empty(FACET.itemsize * C * _CAP, dtype=torch.uint8, device=dev)
    count = torch.empty(C, dtype=torch.int32, device=dev)
    blob = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev)
    _abi.check(_abi.lib.scann_voronoi_neighbors(
        d_lat.data_ptr(), d_x.data_ptr(), d_sa.data_ptr(), d_at.data_ptr(), d_cs.data_ptr(), d_cut.data_ptr(), C,
        1 if allow_pathological else 0, _CAP, slots.data_ptr(), count.data_ptr(), blob.data_ptr(),
        ctypes.c_void_p(host.data_ptr()), status.data_ptr(), ctypes.c_void_p(stream.cuda_stream)),
        "scann_voronoi_neighbors")
    stream.synchronize()
    raw = host.numpy()
    off = raw[:4 * (C + 1)].view(np.int32).copy()
    flags = raw[4 * (C + 1):4 * (2 * C + 1)].view(np.int32).copy()
    rec = raw[head:head + FACET.itemsize * int(off[-1])].view(FACET).copy()
    return off, flags, rec


def voronoi_polyhedra(structs: Sequence, cutoff: float = 13.0, allow_pathological: bool = False) -> List[List[np.ndarray]]:
    """pymatgen ``VoronoiNN(weight="solid_angle", tol=0)``: per structure, per site, the finite facets with solid
    angle > 0 as a structured array (fields ``solid_angle``, ``normalized``, ``distance``, ``site``, ``image`` [3])
    sorted by distance, then site, then image."""
    lats, xs = _arrays(structs)
    nat = np.array([len(X) for X in xs], np.int64)
    sa_off = np.zeros(len(xs) + 1, np.int64)
    np.cumsum(nat, out=sa_off[1:])
    A = int(sa_off[-1])
    if A == 0:
        return [[] for _ in structs]
    lat = np.ascontiguousarray(np.stack(lats).reshape(-1, 9))
    X = np.ascontiguousarray(np.concatenate(xs))
    sid = np.repeat(np.arange(len(xs)), nat)
    tops = np.array([max_cutoff(L) for L in lats])
    cut = np.full(A, float(cutoff))
    result = [None] * A
    todo = np.arange(A)
    while len(todo):
        again = []
        for c0 in range(0, len(todo), _CHUNK):
            atoms = todo[c0:c0 + _CHUNK]
            off, flags, rec = _run(lat, X, sa_off, atoms, cut[atoms], allow_pathological)
            for k, a in enumerate(atoms):
                err = int(flags[k]) & ~_INFINITE
                s, site = int(sid[a]), int(a - sa_off[sid[a]])
                if err:
                    why = "; ".join(m for b, m in _MESSAGES.items() if err & b)
                    raise ValueError(f"structure {s}, site {site}: {why}")
                if flags[k] & _INFINITE and not allow_pathological:
                    if cut[a] >= tops[s]:
                        raise ValueError(f"structure {s}, site {site}: infinite Voronoi facet at the largest cutoff "
                                         f"{cut[a]:.3f} Angstrom")
                    cut[a] = min(2 * cut[a], tops[s] + 0.001)
                    again.append(a)
                    continue
                result[a] = rec[off[k]:off[k + 1]]
        todo = np.array(again, np.int64)
    out = []
    for s in range(len(xs)):
        per = []
        for a in range(int(sa_off[s]), int(sa_off[s + 1])):
            r = result[a]
            img = np.stack([(r["image"] & 1023) - 512, ((r["image"] >> 10) & 1023) - 512,
                            ((r["image"] >> 20) & 1023) - 512], -1).astype(np.int32)
            order = np.lexsort((img[:, 2], img[:, 1], img[:, 0], r["site"], r["distance"]))
            f = np.zeros(len(r), [("solid_angle", "<f8"), ("normalized", "<f8"), ("distance", "<f8"),
                                  ("site", "<i4"), ("image", "<i4", (3,))])
            for name in ("solid_angle", "normalized", "distance", "site"):
                f[name] = r[name][order]
            f["image"] = img[order]
            per.append(f)
        out.append(per)
    return out


def compute_voronoi_neighbors(structs: Sequence, d_thresh: float = 4.0, w_thresh: float = 0.4, cutoff: float = 13.0,
                              allow_pathological: bool = False) -> List[List[List[tuple]]]:
    """``compute_voronoi_neighbor`` over many structures in one pass on the GPU.  Per structure, per atom ``i``, the
    tuples ``(i, site_index, solid_angle, normalized_solid_angle, distance)`` of the facets with ``distance <= d_thresh``
    and normalised solid angle ``>= w_thresh``, sorted by distance, site index, image -- the ``data_neighbor`` format
    of ``DataIterator`` and the ``neighbors=`` argument of ``prepare_input_pmt``."""
    out = []
    for per in voronoi_polyhedra(structs, cutoff, allow_pathological):
        lists = []
        for i, f in enumerate(per):
            sel = f[(f["distance"] <= d_thresh) & (f["normalized"] >= w_thresh)]
            lists.append([(i, int(r["site"]), float(r["solid_angle"]), float(r["normalized"]), float(r["distance"]))
                          for r in sel])
        out.append(lists)
    return out


def compute_voronoi_neighbor(struct, d_thresh: float = 4.0, w_thresh: float = 0.4, cutoff: float = 13.0,
                             allow_pathological: bool = False) -> List[List[tuple]]:
    """The reference's ``compute_voronoi_neighbor(struct, d_thresh, w_thresh)`` for one structure (see
    ``compute_voronoi_neighbors``)."""
    return compute_voronoi_neighbors([struct], d_thresh, w_thresh, cutoff, allow_pathological)[0]
