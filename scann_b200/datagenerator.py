"""``DataIterator`` of the reference (scann/utils/datagenerator.py:12-135) on flat CSR arrays.

The reference rebuilds every padded batch from nested Python lists (three list comprehensions over all
atom-neighbour pairs per ``__getitem__``) -- at 10^5 structures/s on the GPU that host work is the bottleneck.
Here the ragged data are converted ONCE into CSR arrays (structure -> atoms -> neighbours); a batch is either

* ``__getitem__(i)``: the same padded dict ``(inputs, target)`` the reference returns, packed with vectorised
  numpy (bit-identical to the reference's padding, tests/test_datagen.py), or
* ``csr_item(i)``: the CSR slice of the batch, which ``Engine.load_batch_csr`` ships in one host->device copy
  (only valid atoms / pairs travel) and ``scann_pack_batch`` (csrc/plan.cu) expands into the padded device
  buffers.

Data format (reference): ``data_neighbor[s][a]`` = list of neighbour tuples ``n`` with ``n[1]`` = neighbour atom
index, ``n[2]`` = solid angle, ``n[3]`` = normalised solid angle, ``n[-1]`` = distance; ``data_energy[s]`` =
``(atomic numbers, target[, ring/aromatic flags per atom])``.
"""
from __future__ import annotations

from math import ceil
from typing import Dict, Optional, Tuple

import numpy as np


ATOMIC_FEATURES = None      # [Z + 1, 92] float32 table for feature='cgcnn' (set_atomic_features / load_atomic_features)


def set_atomic_features(table) -> np.ndarray:
    """Install the per-element feature vectors ``feature='cgcnn'`` batches are built from -- the reference keeps them
    as ``atomic_features`` (scann/utils/dataset/atomic_data.py: CGCNN's ``atom_init.json``, one 92-vector per atomic
    number, keys are strings, key "0" is the padding atom).  ``table``: such a dict, or an array ``[Z + 1, 92]``.
    The table itself is data of the CGCNN project and is not shipped with this package."""
    global ATOMIC_FEATURES
    arr = _table_array(table)
    if arr.ndim != 2:
        raise ValueError("atomic feature table must be [Z + 1, features]")
    ATOMIC_FEATURES = arr
    return arr


def _table_array(table) -> np.ndarray:
    """A feature table given as CGCNN's ``atom_init.json`` dict (string keys) or as an array -> float32 array."""
    if isinstance(table, dict):
        zmax = max(int(k) for k in table)
        width = len(next(iter(table.values())))
        arr = np.zeros((zmax + 1, width), np.float32)
        for k, v in table.items():
            arr[int(k)] = np.asarray(v, np.float32)
        return arr
    return np.ascontiguousarray(table, np.float32)


def check_atomic_features(table) -> np.ndarray:
    """The per-element feature table of a ``feature='cgcnn'`` model as the device routes read it: a 2-D float32 array
    (or an ``atom_init.json`` dict) with exactly 92 columns, finite, and at least row 0 (padded atoms read row 0, as
    ``DataIterator`` gives them ``ATOMIC_FEATURES[0]``).  Returns it as a C-contiguous float32 array."""
    if isinstance(table, dict):
        arr = _table_array(table)
    else:
        arr = np.asarray(table)
        if arr.dtype != np.float32:
            raise ValueError(f"atomic_features must be float32, not {arr.dtype}")
        arr = np.ascontiguousarray(arr)
    if arr.ndim != 2 or arr.shape[1] != 92 or arr.shape[0] < 1:
        raise ValueError(f"atomic_features must be [Z + 1, 92] (row 0: the padding atom), not {list(arr.shape)}")
    if not np.isfinite(arr).all():
        r = int(np.flatnonzero(~np.isfinite(arr).all(1))[0])
        raise ValueError(f"atomic_features: row {r} holds a value that is not finite")
    return arr


def check_table_rows(z, atom_off, rows: int) -> None:
    """Every atomic number of a data set (``z`` flat, structure s = atoms ``atom_off[s]:atom_off[s + 1]``) has a row in
    a feature table of ``rows`` rows; else ValueError naming the first structure that does not."""
    z = np.asarray(z)
    bad = (z < 0) | (z >= rows)
    if bad.any():
        a = int(np.argmax(bad))
        s = int(np.searchsorted(np.asarray(atom_off), a, side="right")) - 1
        raise ValueError(f"structure {s}: atomic number {int(z[a])} has no row in the atomic feature table "
                         f"({rows} rows, atomic numbers 0..{rows - 1})")


def check_ring_aromatic(ring_aromatic, n_atoms) -> np.ndarray:
    """The ring / aromatic flags of a ``use_ring`` model's structures as the device routes read them: one ``[n_k, 2]``
    array of integers per structure, in order (the third item of a reference ``data_energy`` row, or openbabel's ring
    and aromaticity perception run by the caller), ``n_atoms[k]`` = n_k sites.  The values must fit in int32, the type
    ``DataIterator`` keeps them in.  Returns them concatenated as one C-contiguous int32 array ``[sum(n_k), 2]``;
    else ValueError naming the first structure (its index in ``n_atoms``) whose flags do not fit."""
    n_atoms = [int(n) for n in n_atoms]
    try:
        flags = list(ring_aromatic)
    except TypeError:
        raise ValueError("ring_aromatic must be a sequence of [n_sites, 2] integer arrays, one per structure") from None
    if len(flags) != len(n_atoms):
        raise ValueError(f"{len(n_atoms)} structures but {len(flags)} ring_aromatic arrays")
    out = np.zeros((sum(n_atoms), 2), np.int32)
    a0 = 0
    for k, (f, n) in enumerate(zip(flags, n_atoms)):
        arr = np.asarray(f)
        if arr.shape != (n, 2):
            raise ValueError(f"structure {k}: ring_aromatic must be [{n}, 2] (one row per site), not {list(arr.shape)}")
        if arr.dtype.kind == "f":
            if not (np.isfinite(arr).all() and (arr == np.round(arr)).all()):
                raise ValueError(f"structure {k}: ring_aromatic holds a value that is not an integer")
        elif arr.dtype.kind not in "biu":
            raise ValueError(f"structure {k}: ring_aromatic must hold integers, not {arr.dtype}")
        if arr.size and (arr.min() < -_INT32_MAX - 1 or arr.max() > _INT32_MAX):
            raise ValueError(f"structure {k}: ring_aromatic holds a value outside int32")
        out[a0:a0 + n] = arr
        a0 += n
    return out


def load_atomic_features(path: str) -> np.ndarray:
    """``set_atomic_features`` from a JSON file in CGCNN's ``atom_init.json`` format ({"1": [...], "2": [...], ...})."""
    import json
    with open(path) as f:
        return set_atomic_features(json.load(f))


class DataIterator:
    def __init__(self, data_energy, data_neighbor, batch_size=32, converter=False, use_ring=False, shuffle=False,
                 feature="atomic", g_update=False, atomic_features=None):
        if feature not in ("atomic", "cgcnn"):
            raise ValueError(f"feature must be 'atomic' or 'cgcnn', got {feature!r}")
        if atomic_features is not None:
            set_atomic_features(atomic_features)
        if feature == "cgcnn" and ATOMIC_FEATURES is None:
            raise NotImplementedError("feature='cgcnn' needs the per-element feature table: pass atomic_features= or call "
                                      "scann_b200.datagenerator.load_atomic_features(<atom_init.json>)")
        self.batch_size, self.shuffle, self.use_ring, self.feature = batch_size, shuffle, use_ring, feature
        # the table the cgcnn batches of this iterator are built with (DeviceDataIterator.from_data_iterator takes it)
        self.atomic_features = ATOMIC_FEATURES if feature == "cgcnn" else None
        self.weight_index = 2 if g_update else 3                       # datagenerator.py:48-50
        self.converter = 1000 if converter else 1.0                    # :54-57
        S = len(data_energy)
        n_atoms = np.fromiter((len(c) for c in data_neighbor), np.int64, S)
        self.atom_off = np.zeros(S + 1, np.int64)
        np.cumsum(n_atoms, out=self.atom_off[1:])
        A = int(self.atom_off[-1])
        n_nbr = np.fromiter((len(lc) for c in data_neighbor for lc in c), np.int64, A)
        self.nbr_off = np.zeros(A + 1, np.int64)
        np.cumsum(n_nbr, out=self.nbr_off[1:])
        P = int(self.nbr_off[-1])
        self.nbr_idx = np.fromiter((n[1] for c in data_neighbor for lc in c for n in lc), np.int32, P)
        wi = self.weight_index
        self.nbr_w = np.fromiter((n[wi] for c in data_neighbor for lc in c for n in lc), np.float32, P)
        self.nbr_d = np.fromiter((n[-1] for c in data_neighbor for lc in c for n in lc), np.float32, P)
        self.z = np.fromiter((z for p in data_energy for z in p[0]), np.int32, A)
        self.energy = np.array([float(p[1]) * self.converter for p in data_energy], "float32")
        self.ring = (np.array([r for p in data_energy for r in p[2]], np.int32).reshape(A, 2) if use_ring else None)
        self.on_epoch_end()

    def on_epoch_end(self):
        self.indexes = np.arange(len(self.energy))
        if self.shuffle:
            np.random.shuffle(self.indexes)

    def __len__(self):
        return ceil(len(self.energy) / self.batch_size)

    # ------------------------------------------------------------------ CSR slice of one batch
    def csr_item(self, idx: int) -> Tuple[Dict[str, np.ndarray], np.ndarray]:
        sel = self.indexes[idx * self.batch_size:(idx + 1) * self.batch_size]
        a0, a1 = self.atom_off[sel], self.atom_off[sel + 1]
        n_at = (a1 - a0).astype(np.int64)
        atoms = np.concatenate([np.arange(s, e) for s, e in zip(a0, a1)]) if len(sel) else np.zeros(0, np.int64)
        p0, p1 = self.nbr_off[atoms], self.nbr_off[atoms + 1]
        n_nb = (p1 - p0).astype(np.int64)
        pairs = np.concatenate([np.arange(s, e) for s, e in zip(p0, p1)]) if len(atoms) else np.zeros(0, np.int64)
        sa = np.zeros(len(sel) + 1, np.int32)
        np.cumsum(n_at, out=sa[1:])
        an = np.zeros(len(atoms) + 1, np.int32)
        np.cumsum(n_nb, out=an[1:])
        csr = {"struct_atom_off": sa, "atom_nbr_off": an, "z": self.z[atoms], "nbr_idx": self.nbr_idx[pairs],
               "nbr_w": self.nbr_w[pairs], "nbr_d": self.nbr_d[pairs],
               "M": int(n_at.max()) if len(sel) else 0, "N": int(n_nb.max()) if len(atoms) else 0}
        if self.use_ring:
            csr["ring"] = self.ring[atoms]
        return csr, self.energy[sel]

    # ------------------------------------------------------------------ padded batch, as the reference returns it
    def __getitem__(self, idx: int):
        csr, energy = self.csr_item(idx)
        inputs = pack_padded(csr)
        if self.feature == "cgcnn":        # datagenerator.py:107-110: the mask comes from the atomic numbers, then the
            inputs["atomic"] = ATOMIC_FEATURES[inputs["atomic"]]      # numbers are replaced by their feature vectors
        return inputs, energy


_INT32_MAX = 0x7fffffff
_DEVICE_ARRAYS = ("struct_atom_off", "atom_nbr_off", "z", "nbr_idx", "nbr_w", "nbr_d", "ring", "target")


def _refuse_structures_route(who: str, use_ring: bool, feature: str, atomic_features=None,
                             ring_aromatic=None) -> None:
    if feature == "cgcnn" and atomic_features is None:
        raise NotImplementedError(f"{who}: feature='cgcnn' needs the per-element feature table the model embeds atoms "
                                  "with: pass atomic_features=<[Z + 1, 92] float32 array> (for from_data_iterator: "
                                  "build the DataIterator with atomic_features=)")
    _refuse_ring_route(who, use_ring, ring_aromatic)


def _refuse_ring_route(who: str, use_ring: bool, ring_aromatic) -> None:
    if use_ring and ring_aromatic is None:
        raise NotImplementedError(f"{who}: use_ring models read the ring / aromatic flags of openbabel, which the "
                                  "geometry does not give: pass ring_aromatic=<one [n_sites, 2] integer array per "
                                  "structure> (the third item of the reference's data_energy rows, or openbabel's ring "
                                  "and aromaticity perception run on the structures)")
    if not use_ring and ring_aromatic is not None:
        raise ValueError(f"{who}: ring_aromatic is read by use_ring models only; this one has use_ring=False")


def _check_int32_offsets(atom_off: np.ndarray, pair_off: Optional[np.ndarray] = None) -> None:
    """The device offsets are int32: refuse a data set whose atom or pair offsets reach 2^31, naming the first
    structure that does not fit."""
    for what, off in (("atoms", atom_off), ("neighbour pairs", pair_off)):
        if off is not None and int(off[-1]) > _INT32_MAX:
            s = int(np.searchsorted(off[1:], _INT32_MAX, side="right"))
            raise ValueError(f"structure {s}: the data set's {what} exceed int32 offsets ({int(off[-1])} in all, at most "
                             f"{_INT32_MAX}); split it into data sets below 2^31 {what}")


class DeviceDataIterator:
    """``DataIterator`` with the whole data set resident on the GPU: the CSR arrays and the targets are uploaded once,
    the epoch's shuffle order once per epoch, and ``Engine.load_batch_gather`` pads a batch straight out of them
    (``scann_gather_batch``, csrc/plan.cu).  A training step then copies nothing from the host and does O(batch) host
    work: the batch's M / N / P come from per-structure sizes kept on the host.

    Same Sequence protocol and semantics as ``DataIterator`` (``batch_size``, ``shuffle``, ``converter``,
    ``use_ring``, ``g_update`` -> weight column, ``len``, ``on_epoch_end`` with ``np.random.shuffle`` of the global
    generator): the batches, and the generator's stream, are those of the host iterator.  ``ScannKerasModel.fit`` and
    ``SCANN.evaluate`` take the device route for it; ``csr_item`` / ``__getitem__`` return the host forms of
    ``DataIterator`` (copied back from the device) for any other consumer.

    Build it with ``from_data_iterator`` (the reference's ``.npy`` flow) or ``from_structures`` (Voronoi neighbour
    lists selected on the device; nothing per site reaches the host).

    ``feature='cgcnn'``: the iterator carries the per-element feature table ``atomic_features`` ([Z + 1, 92] float32)
    on the host; the device arrays keep the atomic numbers, and the model embeds them through that table
    (``Engine.set_atomic_features``), so no per-atom feature vector is built.  ``__getitem__`` returns the feature
    vectors ``atomic_features[Z]`` as ``DataIterator.__getitem__`` does."""

    def __init__(self, arrays: Dict[str, object], energy: np.ndarray, atom_off: np.ndarray, pair_off: np.ndarray,
                 nmax: np.ndarray, npairs: np.ndarray, batch_size: int = 32, shuffle: bool = False,
                 use_ring: bool = False, weight_index: int = 3, converter: float = 1.0, indexes=None,
                 feature: str = "atomic", atomic_features=None):
        """Low-level constructor.  ``arrays``: device tensors ``struct_atom_off`` [S+1] / ``atom_nbr_off`` [A+1] (int32,
        from 0), ``z`` [A], ``nbr_idx`` / ``nbr_w`` / ``nbr_d`` [P], ``ring`` [A, 2] int32 or None, ``target`` [S]
        float32.  Host: ``energy`` [S] float32 (the targets), ``atom_off`` / ``pair_off`` [S+1] int64 (first atom /
        pair of each structure), ``nmax`` [S] (longest neighbour list, 1000 entries included) and ``npairs`` [S]
        (entries other than 1000).  ``indexes``: the current epoch order (default: a first ``on_epoch_end``, as
        ``DataIterator`` does).  ``feature='cgcnn'`` needs ``atomic_features`` (``check_atomic_features``)."""
        if feature not in ("atomic", "cgcnn"):
            raise ValueError(f"feature must be 'atomic' or 'cgcnn', got {feature!r}")
        _refuse_structures_route("DeviceDataIterator", False, feature, atomic_features)
        self.batch_size, self.shuffle, self.use_ring, self.feature = batch_size, shuffle, use_ring, feature
        self.atomic_features = check_atomic_features(atomic_features) if feature == "cgcnn" else None
        self.weight_index, self.converter = weight_index, converter
        for k in _DEVICE_ARRAYS:
            setattr(self, k, arrays.get(k))
        self.energy = np.asarray(energy, np.float32)
        self.atom_off, self.pair_off = np.asarray(atom_off, np.int64), np.asarray(pair_off, np.int64)
        self.n_atoms = np.diff(self.atom_off)
        self.nmax, self.npairs = np.asarray(nmax, np.int64), np.asarray(npairs, np.int64)
        self._perm = None
        if indexes is None:
            self.on_epoch_end()
        else:
            self.indexes, self._perm_stale = np.array(indexes, copy=True), True

    # ------------------------------------------------------------------ constructors
    @classmethod
    def from_data_iterator(cls, it: "DataIterator", device=None) -> "DeviceDataIterator":
        """Upload a host ``DataIterator``'s flat arrays once and take over its settings and its current order (and, for
        ``feature='cgcnn'``, the feature table it was built with)."""
        feature = getattr(it, "feature", "atomic")
        table = getattr(it, "atomic_features", None) if feature == "cgcnn" else None
        _refuse_structures_route("DeviceDataIterator.from_data_iterator", False, feature, table)
        atom_off = np.asarray(it.atom_off, np.int64)
        nbr_off = np.asarray(it.nbr_off, np.int64)
        _check_int32_offsets(atom_off, nbr_off[atom_off])
        if table is not None:
            table = check_atomic_features(table)
            check_table_rows(it.z, atom_off, len(table))
        pair_off, nmax, npairs = cls.host_sizes(atom_off, nbr_off, it.nbr_idx)
        from . import _abi
        import torch
        _abi.require_gpu()
        dev = device or torch.device("cuda", torch.cuda.current_device())

        def up(a, dt):
            return torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)
        arrays = {"struct_atom_off": up(atom_off, np.int32), "atom_nbr_off": up(nbr_off, np.int32), "z": up(it.z, np.int32),
                  "nbr_idx": up(it.nbr_idx, np.int32), "nbr_w": up(it.nbr_w, np.float32),
                  "nbr_d": up(it.nbr_d, np.float32), "target": up(it.energy, np.float32),
                  "ring": up(it.ring, np.int32) if it.use_ring else None}
        return cls(arrays, it.energy, atom_off, pair_off, nmax, npairs, batch_size=it.batch_size, shuffle=it.shuffle,
                   use_ring=it.use_ring, weight_index=it.weight_index, converter=it.converter, indexes=it.indexes,
                   feature=feature, atomic_features=table)

    @staticmethod
    def host_sizes(atom_off, nbr_off, nbr_idx):
        """Per-structure host arrays of a data set in ``DataIterator``'s CSR form: ``(pair_off [S+1], nmax [S],
        npairs [S])``, the first pair row, the longest neighbour list (1000 entries included, as ``csr_item``'s ``N``)
        and the entries other than 1000 (as ``load_batch_csr``'s pair count)."""
        atom_off, nbr_off = np.asarray(atom_off, np.int64), np.asarray(nbr_off, np.int64)
        pair_off = nbr_off[atom_off]
        n_nb = np.append(np.diff(nbr_off), 0)
        nmax = np.maximum.reduceat(n_nb, atom_off[:-1]) if len(atom_off) > 1 else np.zeros(0, np.int64)
        nmax[np.diff(atom_off) == 0] = 0
        valid = np.zeros(len(nbr_idx) + 1, np.int64)
        np.cumsum(np.asarray(nbr_idx) != 1000, out=valid[1:])
        return pair_off, nmax, valid[pair_off[1:]] - valid[pair_off[:-1]]

    @classmethod
    def from_structures(cls, structs, targets, batch_size: int = 32, shuffle: bool = False, g_update: bool = True,
                        d_t: float = 4.0, w_t: float = 0.4, angle=None, cutoff: float = 13.0,
                        allow_pathological: bool = False, converter: bool = False, use_ring: bool = False,
                        feature: str = "atomic", atomic_features=None, ring_aromatic=None,
                        device=None) -> "DeviceDataIterator":
        """The iterator ``DataIterator(data_energy, compute_voronoi_neighbors(structs, d_t, w_t), ...)`` would be, with
        the neighbour lists selected and flattened on the device (``voronoi.select_neighbors``, in the chunks of
        ``predict_structures``): no facet record and no neighbour list reaches the host.  ``targets``: one value per
        structure.  ``angle``: the weight column (True = solid angle, False = normalised); None picks the one
        ``DataIterator`` trains a model with this ``g_update`` on.  ``d_t`` / ``w_t`` / ``cutoff`` /
        ``allow_pathological``: as in ``compute_voronoi_neighbors``.  ``feature='cgcnn'`` needs ``atomic_features``, the
        model's per-element feature table ([Z + 1, 92] float32).  ``use_ring=True`` needs ``ring_aromatic``: one
        ``[n_sites, 2]`` integer array per structure (the third item of a ``data_energy`` row; ``check_ring_aromatic``),
        uploaded once as the iterator's ``ring`` array.

        Refused: ``use_ring`` without ``ring_aromatic``, and ``feature='cgcnn'`` without ``atomic_features``
        (``NotImplementedError``); ``ring_aromatic`` without ``use_ring``, flags of the wrong count, shape or values,
        structures without sites, with more than 1000 (1000 is the reference's neighbour padding marker) or, for
        ``feature='cgcnn'``, with an atomic number that has no row in the table (``ValueError``, naming the
        structure)."""
        from . import voronoi as V
        from .model import MAX_STRUCTURE_ATOMS, _structure_chunks
        _refuse_structures_route("DeviceDataIterator.from_structures", use_ring, feature, atomic_features, ring_aromatic)
        if feature == "cgcnn":
            atomic_features = check_atomic_features(atomic_features)
        structs = list(structs)
        targets = list(np.asarray(targets, dtype=object).reshape(-1))
        if len(targets) != len(structs):
            raise ValueError(f"{len(structs)} structures but {len(targets)} targets")
        if batch_size < 1:
            raise ValueError("batch_size must be >= 1")
        lats, xs = V._arrays(structs)
        for k, X in enumerate(xs):
            if len(X) == 0:
                raise ValueError(f"structure {k} has no sites")
            if len(X) > MAX_STRUCTURE_ATOMS:
                raise ValueError(f"structure {k} has {len(X)} sites: at most {MAX_STRUCTURE_ATOMS} (a neighbour index "
                                 "of 1000 is the reference's padding marker and would be masked); train on such "
                                 "structures from host-built batches: compute_voronoi_neighbors + DataIterator")
        n_atoms = np.array([len(X) for X in xs], np.int64)
        atom_off = np.zeros(len(structs) + 1, np.int64)
        np.cumsum(n_atoms, out=atom_off[1:])
        _check_int32_offsets(atom_off)
        if feature == "cgcnn":
            check_table_rows(np.concatenate([np.asarray(s.atomic_numbers).reshape(-1) for s in structs]), atom_off,
                             len(atomic_features))
        ring = check_ring_aromatic(ring_aromatic, n_atoms) if use_ring else None
        conv = 1000 if converter else 1.0
        energy = np.array([float(t) * conv for t in targets], "float32")
        column = bool(g_update) if angle is None else bool(angle)
        import torch
        from . import _abi
        _abi.require_gpu()
        dev = device or torch.device("cuda", torch.cuda.current_device())
        A = int(atom_off[-1])
        an = torch.empty(A + 1, dtype=torch.int32, device=dev)
        z = torch.empty(A, dtype=torch.int32, device=dev)
        parts, nmax, npairs, pbase = [], [], [], 0
        for c0, c1 in _structure_chunks(n_atoms, batch_size):
            sel = V.select_neighbors(structs[c0:c1], d_t, w_t, column, cutoff, allow_pathological, first_index=c0,
                                     _checked=(lats[c0:c1], xs[c0:c1]))
            csr = sel.csr()
            a0, a1 = int(atom_off[c0]), int(atom_off[c1])
            if pbase + csr["P"] > _INT32_MAX:
                s = c0 + int(np.searchsorted(np.cumsum(csr["npairs"]), _INT32_MAX - pbase, side="right"))
                raise ValueError(f"structure {s}: the data set's neighbour pairs exceed int32 offsets (at most "
                                 f"{_INT32_MAX}); split it into data sets below 2^31 pairs")
            an[a0:a1] = csr["atom_nbr_off"][:-1] + pbase      # rebased onto the whole data set's pair rows
            z[a0:a1] = csr["z"]
            parts.append((csr["nbr_idx"].clone(), csr["nbr_w"].clone(), csr["nbr_d"].clone()))
            nmax.append(csr["nmax"])
            npairs.append(csr["npairs"])
            pbase += csr["P"]
        an[A] = pbase
        npairs = np.concatenate(npairs).astype(np.int64)
        pair_off = np.zeros(len(structs) + 1, np.int64)
        np.cumsum(npairs, out=pair_off[1:])

        def cat(k, dt):
            return torch.cat([p[k] for p in parts]) if parts else torch.empty(0, dtype=dt, device=dev)
        arrays = {"struct_atom_off": torch.from_numpy(atom_off.astype(np.int32)).to(dev), "atom_nbr_off": an, "z": z,
                  "nbr_idx": cat(0, torch.int32), "nbr_w": cat(1, torch.float32), "nbr_d": cat(2, torch.float32),
                  "target": torch.from_numpy(energy).to(dev),
                  "ring": torch.from_numpy(ring).to(dev) if use_ring else None}
        return cls(arrays, energy, atom_off, pair_off, np.concatenate(nmax), npairs, batch_size=batch_size,
                   shuffle=shuffle, use_ring=bool(use_ring), weight_index=2 if column else 3, converter=conv,
                   feature=feature, atomic_features=atomic_features)

    # ------------------------------------------------------------------ Sequence protocol
    def on_epoch_end(self):
        self.indexes = np.arange(len(self.energy))                # exactly DataIterator.on_epoch_end
        if self.shuffle:
            np.random.shuffle(self.indexes)
        self._perm_stale = True

    def __len__(self):
        return ceil(len(self.energy) / self.batch_size)

    @property
    def perm(self):
        """The epoch's order on the device (int32 [S]); uploaded with one plain copy after each ``on_epoch_end``."""
        import torch
        if self._perm is None:
            self._perm = torch.empty(len(self.energy), dtype=torch.int32, device=self.struct_atom_off.device)
        if self._perm_stale:
            self._perm.copy_(torch.from_numpy(self.indexes.astype(np.int32)))
            self._perm_stale = False
        return self._perm

    def batch_shape(self, idx: int) -> Tuple[int, int, int, int, int]:
        """``(start, B, M, N, P)`` of batch ``idx``: its first position in the epoch's order, its structures, most
        atoms, longest neighbour list and valid pairs -- the arguments of ``Engine.load_batch_gather``."""
        start = idx * self.batch_size
        sel = self.indexes[start:start + self.batch_size]
        if len(sel) == 0:
            raise IndexError(f"batch {idx} out of range ({len(self)} batches)")
        return (start, len(sel), int(self.n_atoms[sel].max()), int(self.nmax[sel].max()),
                int(self.npairs[sel].sum()))

    def batch_target(self, idx: int) -> np.ndarray:
        return self.energy[self.indexes[idx * self.batch_size:(idx + 1) * self.batch_size]]

    # ------------------------------------------------------------------ host forms (copied back from the device)
    def csr_item(self, idx: int) -> Tuple[Dict[str, np.ndarray], np.ndarray]:
        """``DataIterator.csr_item``: the batch's CSR slice, gathered from the device arrays."""
        import torch
        start, B, M, N, _ = self.batch_shape(idx)
        sel = self.indexes[start:start + B]
        dev = self.struct_atom_off.device
        atoms = np.concatenate([np.arange(self.atom_off[s], self.atom_off[s + 1]) for s in sel])
        pairs = np.concatenate([np.arange(self.pair_off[s], self.pair_off[s + 1]) for s in sel])
        d_atoms = torch.from_numpy(atoms).to(dev)
        d_pairs = torch.from_numpy(pairs).to(dev)
        an = self.atom_nbr_off
        n_nb = (an[d_atoms + 1] - an[d_atoms]).cpu().numpy()
        sa = np.zeros(B + 1, np.int32)
        np.cumsum(self.n_atoms[sel], out=sa[1:])
        ao = np.zeros(len(atoms) + 1, np.int32)
        np.cumsum(n_nb, out=ao[1:])
        csr = {"struct_atom_off": sa, "atom_nbr_off": ao, "z": self.z[d_atoms].cpu().numpy(),
               "nbr_idx": self.nbr_idx[d_pairs].cpu().numpy(), "nbr_w": self.nbr_w[d_pairs].cpu().numpy(),
               "nbr_d": self.nbr_d[d_pairs].cpu().numpy(), "M": M, "N": N}
        if self.use_ring:
            csr["ring"] = self.ring[d_atoms].cpu().numpy()
        return csr, self.energy[sel]

    def __getitem__(self, idx: int):
        """``DataIterator.__getitem__``: the padded batch, gathered by ``scann_gather_batch`` and copied back (for
        ``feature='cgcnn'`` with the atomic numbers replaced by their feature vectors, as ``DataIterator`` does)."""
        inputs, target = self._gathered_item(idx)
        if self.feature == "cgcnn":
            inputs["atomic"] = self.atomic_features[inputs["atomic"]]
        return inputs, target

    def _gathered_item(self, idx: int):
        """The padded batch with atomic numbers, gathered on the device and copied back."""
        import torch
        from ._abi import check, lib
        start, B, M, N, _ = self.batch_shape(idx)
        dev = self.struct_atom_off.device
        i32, f32, u8 = (dict(dtype=t, device=dev) for t in (torch.int32, torch.float32, torch.uint8))
        atomic, amask = torch.empty(B * M, **i32), torch.empty(B * M, **u8)
        nbr, nmask = torch.empty(B * M * N, **i32), torch.empty(B * M * N, **u8)
        w, d = torch.empty(B * M * N, **f32), torch.empty(B * M * N, **f32)
        ring = torch.empty(B * M * 2, **f32) if self.use_ring else None
        tgt = torch.empty(B, **f32)
        perm = self.perm
        check(lib.scann_gather_batch(self.struct_atom_off.data_ptr(), self.atom_nbr_off.data_ptr(), self.z.data_ptr(),
                                     self.nbr_idx.data_ptr(), self.nbr_w.data_ptr(), self.nbr_d.data_ptr(),
                                     self.ring.data_ptr() if self.use_ring else None, self.target.data_ptr(),
                                     perm.data_ptr() + 4 * start, B, M, N, atomic.data_ptr(), amask.data_ptr(),
                                     nbr.data_ptr(), nmask.data_ptr(), w.data_ptr(), d.data_ptr(),
                                     ring.data_ptr() if ring is not None else None, tgt.data_ptr(),
                                     torch.cuda.current_stream(dev).cuda_stream), "gather_batch")
        atomic = atomic.cpu().numpy().reshape(B, M)
        out = {"atomic": atomic, "atom_mask": amask.cpu().numpy().reshape(B, M, 1).astype(bool),
               "neighbors": nbr.cpu().numpy().reshape(B, M, N),
               "neighbor_mask": nmask.cpu().numpy().reshape(B, M, N).astype(bool),
               "neighbor_weight": w.cpu().numpy().reshape(B, M, N), "neighbor_distance": d.cpu().numpy().reshape(B, M, N)}
        if ring is not None:
            out["ring_aromatic"] = ring.cpu().numpy().reshape(B, M, 2).astype(np.int32)
        return out, tgt.cpu().numpy()


def pack_padded(csr: Dict[str, np.ndarray]) -> Dict[str, np.ndarray]:
    """CSR batch -> the padded dict of DataIterator.__getitem__ (vectorised; the device kernel does the same)."""
    sa, an = csr["struct_atom_off"].astype(np.int64), csr["atom_nbr_off"].astype(np.int64)
    B, M, N = len(sa) - 1, csr["M"], csr["N"]
    A = int(sa[-1])
    b_of_atom = np.repeat(np.arange(B), np.diff(sa))
    m_of_atom = np.arange(A) - sa[b_of_atom]
    atomic = np.zeros((B, M), np.int32)
    atomic[b_of_atom, m_of_atom] = csr["z"]
    a_of_pair = np.repeat(np.arange(A), np.diff(an))
    n_of_pair = np.arange(int(an[-1])) - an[a_of_pair]
    bp, mp = b_of_atom[a_of_pair], m_of_atom[a_of_pair]
    nbr = np.zeros((B, M, N), np.int32)
    nmask = np.zeros((B, M, N), bool)
    w = np.zeros((B, M, N), np.float32)
    d = np.zeros((B, M, N), np.float32)
    idx = csr["nbr_idx"]
    nmask[bp, mp, n_of_pair] = idx != 1000          # the reference pads with 1000 and masks "!= 1000" (:82-90)
    nbr[bp, mp, n_of_pair] = np.where(idx == 1000, 0, idx)
    w[bp, mp, n_of_pair] = csr["nbr_w"]
    d[bp, mp, n_of_pair] = csr["nbr_d"]
    out = {"atomic": atomic, "atom_mask": (atomic != 0)[..., None], "neighbors": nbr, "neighbor_mask": nmask,
           "neighbor_weight": w, "neighbor_distance": d}
    if "ring" in csr:
        ring = np.zeros((B, M, 2), np.int32)
        ring[b_of_atom, m_of_atom] = csr["ring"]
        out["ring_aromatic"] = ring
    return out


def pad_sequence(sequences, maxlen=None, dtype="int32", value=0, padding="post"):
    """``pad_sequence`` (scann/utils/general.py:14-32): ``[n, maxlen, ...]`` array filled with ``value``, sequence ``i``
    at the front of row ``i``; a sequence longer than ``maxlen`` keeps its LAST ``maxlen`` items.  ``padding`` is
    accepted and, as in the reference, always behaves as "post"."""
    if maxlen is None:
        maxlen = max(len(seq) for seq in sequences)
    out = np.full((len(sequences), maxlen) + np.asarray(sequences[0]).shape[1:], value, dtype=dtype)
    for row, seq in zip(out, sequences):
        kept = np.asarray(seq[-maxlen:], dtype=dtype)
        row[:len(kept)] = kept
    return out


def pad_nested_sequences(sequences, max_len_1, max_len_2, dtype="int32", value=0):
    """``pad_nested_sequences`` (scann/utils/general.py:35-50): ragged ``[structure][atom][neighbour]`` lists ->
    ``[n, max_len_2 atoms, max_len_1 neighbours]`` filled with ``value``."""
    out = np.full((len(sequences), max_len_2, max_len_1), value, dtype=dtype)
    for block, atoms in zip(out, sequences):
        for row, items in zip(block, atoms[-max_len_2:]):
            kept = np.asarray(items[-max_len_1:], dtype=dtype)
            row[:len(kept)] = kept
    return out


def split_data(len_data, test_percent=0.1, train_size=None, test_size=None):
    """``split_data`` (scann/utils/general.py:79-101): ONE permutation of the global numpy generator (the same
    ``np.random.seed`` gives the reference's split) cut into train | valid | test | extra.  Sizes: the given
    ``train_size`` / ``test_size``, else ``int(len * (1 - 2 * test_percent))`` / ``int(len * test_percent)``; the
    validation set takes what is left."""
    if train_size:
        n_train, n_test = train_size, test_size
    else:
        n_train, n_test = int(len_data * (1 - test_percent * 2)), int(len_data * test_percent)
    n_valid = len_data - n_train - n_test
    order = np.random.permutation(len_data)
    train, valid, test, extra = np.split(order, np.cumsum([n_train, n_valid, n_test]))
    return train, valid, test, extra


def load_dataset(dataset, dataset_neighbor, target_prop, use_ref=False, use_ring=True):
    """``load_dataset`` (scann/utils/general.py:104-144): the pickled object arrays the reference's preprocessing
    writes.  ``dataset``: records ``{"Atomic": [...], "Properties": {name: value, ...}, "Features": {name: per-atom
    flags}}``; ``dataset_neighbor``: the per-structure neighbour lists.  Returns ``(data_energy, data_neighbor)`` as
    object arrays: rows ``[atomic numbers, target, ring/aromatic flags [atoms, n_features]]`` with ``use_ring``
    (which takes precedence), ``[atomic numbers, target - Ref_energy]`` with ``use_ref``, else
    ``[atomic numbers, target]``."""
    records = np.load(dataset, allow_pickle=True)
    if use_ref:
        print("Using reference energy optimization", "\n")
    if use_ring:
        print("Using ring aromatic information", "\n")
    rows = []
    for rec in records:
        value = float(rec["Properties"][target_prop])
        if use_ring:
            rows.append([rec["Atomic"], value, np.stack([rec["Features"][k] for k in rec["Features"]], -1)])
        elif use_ref:
            rows.append([rec["Atomic"], value - float(rec["Properties"]["Ref_energy"])])
        else:
            rows.append([rec["Atomic"], value])
    data_energy = np.array(rows, dtype="object")
    data_neighbor = np.array(np.load(dataset_neighbor, allow_pickle=True), dtype="object")
    return data_energy, data_neighbor


def prepare_input_from_neighbors(atomic_numbers, neighbors, angle: bool = True) -> Dict[str, np.ndarray]:
    """The padding half of ``prepare_input_pmt`` (scann/utils/general.py:218-246) for a caller who already has the
    neighbour lists of ONE structure -- the README inference flow (README.md:102-120) without pymatgen:
    ``neighbors[a]`` = list of tuples ``n`` as ``compute_voronoi_neighbor`` returns them (``n[1]`` neighbour atom
    index, ``n[2]`` solid angle, ``n[3]`` normalised solid angle, ``n[-1]`` distance).  ``angle=True`` selects the raw
    solid angle (what the g_update models are trained on, general.py:224).  Returns the model's input dict with a
    leading batch axis of 1; padded slots carry index 0 / weight 0 / distance 0 and ``neighbor_mask`` False, exactly
    as ``pad_sequence(..., value=1000)`` + ``!= 1000`` produce them (tests/test_reference_pins.py)."""
    na = len(neighbors)
    if len(atomic_numbers) != na:
        raise ValueError("one neighbour list per atom is required")
    n_max = max((len(lc) for lc in neighbors), default=0)
    nbr = np.full((1, na, n_max), 1000, np.int32)
    w = np.zeros((1, na, n_max), np.float32)
    d = np.zeros((1, na, n_max), np.float32)
    wi = 2 if angle else 3
    for a, lc in enumerate(neighbors):
        k = len(lc)
        if k:
            nbr[0, a, :k] = [n[1] for n in lc]
            w[0, a, :k] = [n[wi] for n in lc]
            d[0, a, :k] = [n[-1] for n in lc]
    mask = nbr != 1000
    nbr[nbr == 1000] = 0
    atomics = np.array([atomic_numbers], "int32")
    return {"atomic": atomics, "atom_mask": np.expand_dims(atomics != 0, -1), "neighbors": nbr, "neighbor_mask": mask,
            "neighbor_weight": w, "neighbor_distance": d}


def prepare_input_pmt(struct, d_t=4.0, w_t=0.4, angle=True, neighbors=None) -> Dict[str, np.ndarray]:
    """``prepare_input_pmt`` (scann/utils/general.py:206-246) with the reference's signature.  The Voronoi neighbour
    search behind it (``compute_voronoi_neighbor``: pymatgen + Qhull) is outside this package, so the caller hands the
    neighbour lists over as ``neighbors`` (what ``compute_voronoi_neighbor(struct, d_thresh=d_t, w_thresh=w_t)`` of the
    reference returns); ``struct`` only has to offer ``atomic_numbers``.  Without ``neighbors`` the call fails loudly."""
    if neighbors is None:
        raise NotImplementedError("prepare_input_pmt: the Voronoi neighbour search (pymatgen / Qhull) is not part of the "
                                  "accelerated package; pass neighbors=compute_voronoi_neighbor(struct, d_thresh=d_t, "
                                  "w_thresh=w_t) or call prepare_input_from_neighbors(atomic_numbers, neighbors)")
    return prepare_input_from_neighbors(list(struct.atomic_numbers), neighbors, angle=angle)


def padded_to_csr(inputs: Dict[str, np.ndarray]) -> Dict[str, np.ndarray]:
    """Inverse of ``pack_padded`` for batches whose valid atoms / neighbour slots are prefixes (what
    DataIterator.__getitem__ produces): padded dict -> CSR batch for ``Engine.load_batch_csr``."""
    am = inputs["atom_mask"][..., 0].astype(bool)
    nm = inputs["neighbor_mask"].astype(bool)
    B, M, N = nm.shape
    n_at = am.sum(1)
    if not (np.array_equal(am, np.arange(M)[None, :] < n_at[:, None])):
        raise ValueError("valid atoms must be a prefix of every structure")
    n_nb = nm.sum(2)
    if not np.array_equal(nm, np.arange(N)[None, None, :] < n_nb[..., None]):
        raise ValueError("valid neighbour slots must be a prefix of every atom")
    sa = np.zeros(B + 1, np.int32)
    np.cumsum(n_at, out=sa[1:])
    cnt = n_nb[am]
    an = np.zeros(len(cnt) + 1, np.int32)
    np.cumsum(cnt, out=an[1:])
    sel = nm & am[..., None]
    csr = {"struct_atom_off": sa, "atom_nbr_off": an, "z": inputs["atomic"][am].astype(np.int32),
           "nbr_idx": inputs["neighbors"][sel].astype(np.int32), "nbr_w": inputs["neighbor_weight"][sel].astype(np.float32),
           "nbr_d": inputs["neighbor_distance"][sel].astype(np.float32), "M": M, "N": N}
    if "ring_aromatic" in inputs:
        csr["ring"] = inputs["ring_aromatic"][am].astype(np.int32)
    return csr


def synthetic_ragged(n_struct: int, seed: int = 0, max_atoms: int = 29, max_nbr: int = 16, use_ring: bool = False):
    """Random data in the reference's nested-list format (for tests and benchmarks)."""
    rng = np.random.default_rng(seed)
    data_energy, data_neighbor = [], []
    for _ in range(n_struct):
        na = int(rng.integers(2, max_atoms + 1))
        zs = rng.choice([1, 6, 7, 8, 9], size=na).tolist()
        rec = [zs, float(rng.standard_normal())]
        if use_ring:
            rec.append(rng.integers(0, 2, size=(na, 2)).tolist())
        data_energy.append(tuple(rec))
        nb = []
        for _a in range(na):
            k = int(rng.integers(1, max_nbr + 1))
            nb.append([(0, int(rng.integers(0, na)), float(rng.uniform(0.4, 3.0)), float(rng.uniform(0.2, 1.0)),
                        float(rng.uniform(0.9, 4.0))) for _ in range(k)])
        data_neighbor.append(nb)
    de = np.empty(n_struct, object)
    dn = np.empty(n_struct, object)
    for i in range(n_struct):
        de[i], dn[i] = data_energy[i], data_neighbor[i]
    return de, dn
