"""Voronoi neighbour lists on the GPU: the reference's ``compute_voronoi_neighbor`` (scann/utils/voronoi_neighbor.py:11-61)
without pymatgen.

The reference calls pymatgen's ``VoronoiNN(weight="solid_angle").get_voronoi_polyhedra`` per site (one Qhull
tessellation of every periodic image within ``cutoff``) and keeps the facets within ``d_thresh`` whose solid angle,
normalised by the site's largest, is at least ``w_thresh``.  Here every site of every structure is one warp of
``scann_voronoi_neighbors`` (csrc/voronoi.cu, fp64); pymatgen's retry loop -- a site whose cell still has an unbounded
facet is run again with ``cutoff = min(2 cutoff, longest cell diagonal + 0.011)`` -- re-launches only those sites.
The cell search holds 64 facets; a site whose cell overflows it (a surface atom that sees a slab's periodic images
across the vacuum) runs again, at the same cutoff, in the wide form of 256 facets, and stays wide through later retries.

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
_CAP = 64                       # facet records per centre of the narrow cell search (its facet capacity)
_CAP_WIDE = 256                 # ... of the wide one, for the centres whose cell overflows the narrow one
_CHUNK = 1 << 16                # centres per narrow launch
_CHUNK_WIDE = _CHUNK * _CAP // _CAP_WIDE    # centres per wide launch: the same bytes of facet slots
FACET = np.dtype([("solid_angle", "<f8"), ("normalized", "<f8"), ("distance", "<f8"), ("site", "<i4"),
                  ("image", "<i4")])
_MESSAGES = {ERR_COINCIDENT: "two points of its Voronoi point set are closer than 1e-8 Angstrom",
             ERR_CAPACITY: "its Voronoi cell exceeds the kernel's capacity (256 facets, 64 vertices per facet, 128 "
                           "points in one distance shell, images up to 511 cells away)",
             ERR_NO_FACET: "its Voronoi cell has no finite facet",
             ERR_TOPOLOGY: "a cut of its Voronoi cell was numerically inconsistent"}
# a capacity error together with another error bit in the narrow pass (not retried wide)
_CAPACITY_NARROW = ("its Voronoi cell exceeds the kernel's capacity (64 facets, 32 vertices per facet, 128 points in "
                    "one distance shell, images up to 511 cells away)")


def _why(err, wide):
    return "; ".join(_CAPACITY_NARROW if b == ERR_CAPACITY and not wide else m
                     for b, m in _MESSAGES.items() if err & b)


def _passes(todo, wide):
    """The launches of one round of the retry loop: (centres, cap, wide) for the narrow centres of ``todo``, in
    chunks of ``_CHUNK``, then for its wide ones, in chunks of ``_CHUNK_WIDE``.  A list, split before the first launch:
    a centre that overflows the narrow form in this round is marked wide for the next round, not added to this one."""
    out = []
    for w, cap, chunk in ((False, _CAP, _CHUNK), (True, _CAP_WIDE, _CHUNK_WIDE)):
        part = todo[wide[todo] == w]
        out += [(part[c0:c0 + chunk], cap, w) for c0 in range(0, len(part), chunk)]
    return out


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


def _run(lat, X, sa_off, atoms, cut, allow_pathological, cap=_CAP):
    """One launch over the listed centres with ``cap`` facet slots each (<= 64: the narrow cell search, up to 256: the
    wide one) -> (off [C+1], flags [C], records)."""
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
    nbytes = head + FACET.itemsize * C * cap
    slots = torch.empty(FACET.itemsize * C * cap, dtype=torch.uint8, device=dev)
    count = torch.empty(C, dtype=torch.int32, device=dev)
    blob = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev)
    _abi.check(_abi.lib.scann_voronoi_neighbors(
        d_lat.data_ptr(), d_x.data_ptr(), d_sa.data_ptr(), d_at.data_ptr(), d_cs.data_ptr(), d_cut.data_ptr(), C,
        1 if allow_pathological else 0, cap, slots.data_ptr(), count.data_ptr(), blob.data_ptr(),
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
    wide = np.zeros(A, bool)
    todo = np.arange(A)
    while len(todo):
        again = []
        for atoms, cap, is_wide in _passes(todo, wide):
            off, flags, rec = _run(lat, X, sa_off, atoms, cut[atoms], allow_pathological, cap)
            for k, a in enumerate(atoms):
                err = int(flags[k]) & ~_INFINITE
                s, site = int(sid[a]), int(a - sa_off[sid[a]])
                if err == ERR_CAPACITY and not is_wide:   # the cell overflows the narrow form: again, wide
                    wide[a] = True
                    again.append(a)
                    continue
                if err:
                    raise ValueError(f"structure {s}, site {site}: {_why(err, is_wide)}")
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


# ------------------------------------------------------------------------------------------ neighbour lists on the device
# The same lists as compute_voronoi_neighbors + DataIterator, without the facet records leaving the device:
# scann_voronoi_select orders and thresholds each centre's records into per-atom staging rows, and
# scann_voronoi_batch_csr writes any run of structures as the CSR batch that Engine.load_batch_device_csr packs.
# Only the per-centre flags (retry / error) and a few sizes per batch come back to the host.
_SEL = 64                       # staging slots per atom row: the most neighbours an atom keeps
_ALIGN = 16

# optional CUDA-event log (tools/structure_predict_bench.py): name -> list of (start, end) event pairs
event_log = None


def _timed(name, stream, fn):
    if event_log is None:
        return fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    out = fn()
    e1.record(stream)
    event_log.setdefault(name, []).append((e0, e1))
    return out


class NeighborSelection:
    """Selected neighbour lists of a run of structures, resident on the device (``select_neighbors``): per atom row up
    to 64 ``(site, weight, distance)`` in the order of ``compute_voronoi_neighbors``.  ``csr(s0, s1)`` writes
    structures ``s0 .. s1 - 1`` as one CSR batch."""

    def __init__(self, sa_off, d_sa, d_z, count, idx, w, d):
        self.struct_atom_off = sa_off            # host, int64 [S+1]
        self._d_sa, self._d_z = d_sa, d_z
        self.sel_count, self.sel_idx, self.sel_w, self.sel_d = count, idx, w, d

    def __len__(self):
        return len(self.struct_atom_off) - 1

    def csr(self, s0: int = 0, s1: int = None, ring: torch.Tensor = None) -> dict:
        """Structures ``s0 .. s1 - 1`` as the CSR batch of ``DataIterator.csr_item`` in ONE device blob (``"blob"``,
        byte offsets ``"offsets"``; device views ``struct_atom_off``, ``atom_nbr_off``, ``z``, ``nbr_idx``, ``nbr_w``,
        ``nbr_d``).  Host side: ``B``, ``M`` (most atoms), ``N`` (most kept neighbours), ``P`` (kept pairs) and per
        structure ``n_atoms``, ``nmax``, ``npairs``.

        ``ring``: the ring / aromatic flags of every atom row of the selection, a device int32 tensor ``[A, 2]``.  The
        rows of the batch's atoms (contiguous) are copied into a ``"ring"`` segment of the blob (view ``ring`` [nA, 2]),
        which ``Engine.load_batch_device_csr`` packs like ``DataIterator.csr_item``'s ``ring``."""
        s1 = len(self) if s1 is None else s1
        B = s1 - s0
        sa = self.struct_atom_off
        a0, nA = int(sa[s0]), int(sa[s1] - sa[s0])
        dev = self.sel_count.device
        if ring is not None and (ring.dtype != torch.int32 or ring.device != dev or
                                 tuple(ring.shape) != (int(sa[-1]), 2) or not ring.is_contiguous()):
            raise ValueError(f"ring must be a contiguous int32 tensor [{int(sa[-1])}, 2] on {dev}, not "
                             f"{ring.dtype} {list(ring.shape)} on {ring.device}")
        sizes_b = [("sa", 4 * (B + 1)), ("an", 4 * (nA + 1)), ("z", 4 * nA), ("idx", 4 * nA * _SEL), ("w", 4 * nA * _SEL),
                   ("d", 4 * nA * _SEL)] + ([("ring", 8 * nA)] if ring is not None else [])
        offs, off = {}, 0
        for name, nb in sizes_b:
            offs[name] = off
            off += (nb + _ALIGN - 1) // _ALIGN * _ALIGN
        blob = torch.empty(max(off, _ALIGN), dtype=torch.uint8, device=dev)
        sizes = torch.empty(2 * B, dtype=torch.int32, device=dev)
        stream = torch.cuda.current_stream(dev)
        _timed("voronoi_batch_csr", stream, lambda: _abi.check(_abi.lib.scann_voronoi_batch_csr(
            self._d_sa.data_ptr(), self._d_z.data_ptr(), s0, B, a0, nA, self.sel_count.data_ptr(),
            self.sel_idx.data_ptr(), self.sel_w.data_ptr(), self.sel_d.data_ptr(), blob.data_ptr(), offs["sa"],
            offs["an"], offs["z"], offs["idx"], offs["w"], offs["d"], sizes.data_ptr(),
            ctypes.c_void_p(stream.cuda_stream)), "scann_voronoi_batch_csr"))
        if ring is not None:            # one device-to-device copy on the same stream
            blob[offs["ring"]:offs["ring"] + 8 * nA].view(torch.int32).copy_(ring[a0:a0 + nA].reshape(-1))
        host = torch.empty(2 * B, dtype=torch.int32, pin_memory=True)
        host.copy_(sizes, non_blocking=True)
        stream.synchronize()
        h = host.numpy()
        nmax, npairs = h[:B].copy(), h[B:].copy()
        n_atoms = np.diff(sa[s0:s1 + 1])
        P = int(npairs.sum())

        def view(name, dt, n):
            return blob[offs[name]:offs[name] + 4 * n].view(dt)
        out = {"blob": blob, "offsets": offs, "B": B, "M": int(n_atoms.max()), "N": int(nmax.max()), "P": P,
               "n_atoms": n_atoms, "nmax": nmax, "npairs": npairs,
               "struct_atom_off": view("sa", torch.int32, B + 1), "atom_nbr_off": view("an", torch.int32, nA + 1),
               "z": view("z", torch.int32, nA), "nbr_idx": view("idx", torch.int32, P),
               "nbr_w": view("w", torch.float32, P), "nbr_d": view("d", torch.float32, P)}
        if ring is not None:
            out["ring"] = view("ring", torch.int32, 2 * nA).view(nA, 2)
        return out


def _select_pass(d_lat, d_x, d_sa, sa_off, atoms, cut, allow_pathological, d_t, w_t, column, sel, cap=_CAP):
    """One cell search over the listed centres (``cap`` as in ``_run``), its records thresholded into the staging rows
    -> (flags [C], kept [C] or None) on the host.  ``kept``: the true kept count of every centre, returned only when a
    centre keeps more neighbours than a staging row holds."""
    dev = d_x.device
    C = len(atoms)
    cs = np.searchsorted(sa_off, atoms, side="right") - 1
    # one upload of the per-centre inputs: atom rows, structures (int32), cutoffs (float64, 8-byte aligned after 2C ints)
    head = np.empty(2 * C, np.int32)
    head[:C], head[C:] = atoms, cs
    up = torch.from_numpy(np.concatenate([head.view(np.uint8), np.ascontiguousarray(cut, np.float64).view(np.uint8)]))
    d_up = up.to(dev)
    d_at, d_cs = d_up[:4 * C].view(torch.int32), d_up[4 * C:8 * C].view(torch.int32)
    d_cut = d_up[8 * C:].view(torch.float64)
    hb = (4 * (2 * C + 1) + 31) // 32 * 32
    slots = torch.empty(FACET.itemsize * C * cap, dtype=torch.uint8, device=dev)
    count = torch.empty(C, dtype=torch.int32, device=dev)
    blob = torch.empty(hb + FACET.itemsize * C * cap, dtype=torch.uint8, device=dev)
    status = torch.zeros(2, dtype=torch.int32, device=dev)       # [0]: the cell search, [1]: the select
    stream = torch.cuda.current_stream(dev)
    st = ctypes.c_void_p(stream.cuda_stream)
    wide = "_wide" if cap > _CAP else ""
    _timed("voronoi_neighbors" + wide, stream, lambda: _abi.check(_abi.lib.scann_voronoi_neighbors(
        d_lat.data_ptr(), d_x.data_ptr(), d_sa.data_ptr(), d_at.data_ptr(), d_cs.data_ptr(), d_cut.data_ptr(), C,
        1 if allow_pathological else 0, cap, slots.data_ptr(), count.data_ptr(), blob.data_ptr(), None,
        status.data_ptr(), st), "scann_voronoi_neighbors"))
    count_, idx, w, d = sel
    _timed("voronoi_select" + wide, stream, lambda: _abi.check(_abi.lib.scann_voronoi_select(
        blob.data_ptr(), d_at.data_ptr(), C, float(d_t), float(w_t), 0 if column else 1, count_.data_ptr(),
        idx.data_ptr(), w.data_ptr(), d.data_ptr(), status.data_ptr() + 4, st), "scann_voronoi_select"))
    host = torch.empty(C + 2, dtype=torch.int32, pin_memory=True)
    host[:C].copy_(blob[4 * (C + 1):4 * (2 * C + 1)].view(torch.int32), non_blocking=True)
    host[C:].copy_(status, non_blocking=True)
    stream.synchronize()
    h = host.numpy()
    kept = None
    if h[C + 1] & ERR_CAPACITY:         # more kept neighbours than a staging row holds (or a malformed blob)
        kept = count_[torch.from_numpy(np.asarray(atoms, np.int64)).to(dev)].cpu().numpy()
        if not (kept > _SEL).any():
            raise _abi.ScannAbiError("scann_voronoi_select: a centre has more records than the select accepts")
    return h[:C].copy(), kept


def select_neighbors(structs: Sequence, d_thresh: float = 4.0, w_thresh: float = 0.4, angle: bool = True,
                     cutoff: float = 13.0, allow_pathological: bool = False, first_index: int = 0,
                     _checked=None) -> NeighborSelection:
    """``compute_voronoi_neighbors`` kept on the device: the cell search of every site, pymatgen's retry loop (only the
    per-site flags come back; flagged sites run again with a wider cutoff, their records replace the first ones), then
    the selection of ``scann_voronoi_select``.  ``angle`` picks the weight column as ``prepare_input_pmt`` does: True =
    solid angle, False = normalised solid angle.  Atomic numbers come from ``struct.atomic_numbers``.  A bad structure
    raises the ``ValueError`` of ``voronoi_polyhedra``, numbered ``first_index + k``."""
    _abi.require_gpu()
    lats, xs = _checked if _checked is not None else _arrays(structs)
    dev = torch.device("cuda", torch.cuda.current_device())
    nat = np.array([len(X) for X in xs], np.int64)
    sa_off = np.zeros(len(xs) + 1, np.int64)
    np.cumsum(nat, out=sa_off[1:])
    A = int(sa_off[-1])
    z = np.fromiter((int(v) for st in structs for v in st.atomic_numbers), np.int32) if A else np.zeros(0, np.int32)
    if len(z) != A:
        raise ValueError("every structure needs one atomic number per site (struct.atomic_numbers)")
    sel = (torch.zeros(A, dtype=torch.int32, device=dev), torch.empty(A * _SEL, dtype=torch.int32, device=dev),
           torch.empty(A * _SEL, dtype=torch.float32, device=dev), torch.empty(A * _SEL, dtype=torch.float32, device=dev))
    d_sa = torch.from_numpy(sa_off.astype(np.int32)).to(dev)
    d_z = torch.from_numpy(z).to(dev)
    out = NeighborSelection(sa_off, d_sa, d_z, *sel)
    if A == 0:
        return out
    d_lat = torch.from_numpy(np.ascontiguousarray(np.stack(lats).reshape(-1, 9))).to(dev)
    d_x = torch.from_numpy(np.ascontiguousarray(np.concatenate(xs))).to(dev)
    sid = np.repeat(np.arange(len(xs)), nat)
    tops = np.array([max_cutoff(L) for L in lats])
    cut = np.full(A, float(cutoff))
    wide = np.zeros(A, bool)
    todo = np.arange(A)
    while len(todo):
        again = []
        for atoms, cap, is_wide in _passes(todo, wide):
            flags, kept = _select_pass(d_lat, d_x, d_sa, sa_off, atoms, cut[atoms], allow_pathological, d_thresh,
                                       w_thresh, angle, sel, cap)
            for k in np.flatnonzero(flags):         # the checks of voronoi_polyhedra, in the same order
                a = int(atoms[k])
                err = int(flags[k]) & ~_INFINITE
                s, site = int(sid[a]), int(a - sa_off[sid[a]])
                if err == ERR_CAPACITY and not is_wide:
                    wide[a] = True
                    again.append(a)
                    continue
                if err:
                    raise ValueError(f"structure {first_index + s}, site {site}: {_why(err, is_wide)}")
                if not allow_pathological:
                    if cut[a] >= tops[s]:
                        raise ValueError(f"structure {first_index + s}, site {site}: infinite Voronoi facet at the "
                                         f"largest cutoff {cut[a]:.3f} Angstrom")
                    cut[a] = min(2 * cut[a], tops[s] + 0.001)
                    again.append(a)
            if kept is not None:                    # a centre whose cell is final keeps more than a row holds
                for k in np.flatnonzero(kept > _SEL):
                    a = int(atoms[k])
                    if a in again:
                        continue
                    s, site = int(sid[a]), int(a - sa_off[sid[a]])
                    raise ValueError(f"structure {first_index + s}, site {site}: {int(kept[k])} neighbours kept "
                                     f"(distance <= {d_thresh}, normalised solid angle >= {w_thresh}), more than the "
                                     f"{_SEL} a neighbour list holds")
        todo = np.array(again, np.int64)
    return out


def neighbor_csr(structs: Sequence, d_t: float = 4.0, w_t: float = 0.4, angle: bool = True, cutoff: float = 13.0,
                 allow_pathological: bool = False) -> dict:
    """All ``structs`` as one CSR batch on the device: what ``DataIterator(..., g_update=angle).csr_item`` builds from
    ``compute_voronoi_neighbors(structs, d_t, w_t)``, bit for bit, without the per-site host work (see
    ``NeighborSelection.csr`` for the keys)."""
    return select_neighbors(structs, d_t, w_t, angle, cutoff, allow_pathological).csr()
