"""Drop-in surface of the reference for the accelerated path.

``SCANN(config, pretrained=..., mode=...)`` mirrors scann/models/scann_model.py:42-96 and
``SCANN.model`` mirrors the subset of ``tf.keras.Model`` the reference calls:
``predict`` (:266, :316), ``compile`` (:210-214), ``fit`` (:232-241), ``get_layer`` (:81),
``summary`` (:324, :451) plus ``train_on_batch`` / ``save_weights`` / ``load_weights``.
Arithmetic runs in the sm_100a kernels behind ``libscann_b200.so``; there is no CPU fallback.
"""
from __future__ import annotations

import functools
import math
import os
from typing import Dict, Iterable, NamedTuple, Optional

import numpy as np
import torch

from .config import ModelSpec, fill_cli_defaults, model_spec
from .engine import Batch, Engine
from .params import ParamLayout


# --------------------------------------------------------------------------- lr schedules
class CosineDecay:
    """tf.keras.optimizers.schedules.CosineDecay(lr, decay_steps, alpha) (scann_model.py:203-208)."""

    def __init__(self, initial_learning_rate: float, decay_steps: float, alpha: float = 0.0):
        self.lr0, self.decay_steps, self.alpha = float(initial_learning_rate), float(decay_steps), float(alpha)

    def __call__(self, step: int) -> float:
        s = min(float(step), self.decay_steps)
        cos = 0.5 * (1.0 + math.cos(math.pi * s / self.decay_steps))
        return self.lr0 * ((1.0 - self.alpha) * cos + self.alpha)


class History:
    def __init__(self):
        self.history: Dict[str, list] = {}

    def add(self, key: str, v: float) -> None:
        self.history.setdefault(key, []).append(float(v))


MAX_STRUCTURE_ATOMS = 1000      # predict_structures: a site index of 1000 would read as the padding marker
_CHUNK_ATOMS = 1 << 16          # predict_structures: sites whose neighbour lists are staged on the device at once


def shape_class(M: int, N: int):
    """Padded (M, N) of a ``predict_structures`` batch: atoms up to a multiple of 8; neighbours up to a multiple of 4
    while <= 32 (a batch within 32 keeps the pipelined 32-row plan), else of 8 (at most 64, the facet capacity)."""
    M = max(8, (M + 7) // 8 * 8)
    N = max(4, (N + 3) // 4 * 4) if N <= 32 else (N + 7) // 8 * 8
    return M, N


def _structure_chunks(n_atoms, batch_size: int):
    """Runs of whole batches with about _CHUNK_ATOMS sites (at least one batch): [(first, end)]."""
    out, c0, atoms = [], 0, 0
    for s0 in range(0, len(n_atoms), batch_size):
        s1 = min(s0 + batch_size, len(n_atoms))
        n = sum(n_atoms[s0:s1])
        if s0 > c0 and atoms + n > _CHUNK_ATOMS:
            out.append((c0, s0))
            c0, atoms = s0, 0
        atoms += n
    if c0 < len(n_atoms):
        out.append((c0, len(n_atoms)))
    return out


class LocalAttentionScores(NamedTuple):
    """Local-attention scores of one structure (``predict_structures(..., local_attention=True)``).  Pairs
    ``site_offsets[i]:site_offsets[i + 1]`` are the kept neighbours of site i in the order of
    ``compute_voronoi_neighbor``'s list for that site: site ``neighbors[p]`` at ``distances[p]`` (so periodic images of
    one site stay apart).  ``scores[l, h, p]`` is the weight of pair p in head h of local-attention layer l."""
    site_offsets: np.ndarray        # int32 [n + 1]
    neighbors: np.ndarray           # int32 [P_s]
    distances: np.ndarray           # float32 [P_s]
    scores: np.ndarray              # float32 [n_attention, num_head, P_s]


def split_pair_scores(struct_atom_off, atom_nbr_off, nbr_idx, nbr_d, scores):
    """The [L, 8, P] scores of one CSR batch (``Engine.predict_step(..., local_attention="csr")``, trimmed to its P
    pairs) and the batch's CSR arrays -> one ``LocalAttentionScores`` per structure."""
    sa = np.asarray(struct_atom_off, np.int64)
    an = np.asarray(atom_nbr_off, np.int64)
    scores = np.asarray(scores, np.float32)
    if sa.ndim != 1 or len(sa) < 1 or an.ndim != 1 or len(an) != sa[-1] - sa[0] + 1:
        raise ValueError("struct_atom_off [B+1] and atom_nbr_off [A+1] do not describe one CSR batch")
    P = int(an[-1] - an[0])
    if scores.ndim != 3 or scores.shape[2] != P or len(nbr_idx) < P or len(nbr_d) < P:
        raise ValueError(f"scores {scores.shape}, {len(nbr_idx)} neighbours and {len(nbr_d)} distances for {P} pairs")
    idx, d = np.asarray(nbr_idx, np.int32), np.asarray(nbr_d, np.float32)
    a = (sa - sa[0]).tolist()
    p = (an[sa - sa[0]] - an[0]).tolist()
    off = (an - an[0]).astype(np.int32)
    # views into the batch's arrays (one allocation per structure: its site offsets)
    return [LocalAttentionScores(off[a[s]:a[s + 1] + 1] - off[a[s]], idx[p[s]:p[s + 1]], d[p[s]:p[s + 1]],
                                 scores[:, :, p[s]:p[s + 1]]) for s in range(len(a) - 1)]


def _check_flag(name: str, value) -> bool:
    if not isinstance(value, (bool, np.bool_)):
        raise TypeError(f"{name} must be a bool, not {type(value).__name__}")
    return bool(value)


def _batch_errors(y, y_true) -> Dict[str, float]:
    """MAE / RMSE of one batch's predictions (``evaluate_batch``)."""
    y = np.asarray(y).reshape(-1)
    t = np.asarray(y_true, np.float32).reshape(-1)
    return {"mae": float(np.abs(y - t).mean()), "rmse": float(np.sqrt(((y - t) ** 2).mean()))}


def _ragged_capable(seq) -> bool:
    """A Sequence whose batches may travel as CSR slices: this package's DataIterator on atomic-number features
    (cgcnn batches carry per-atom feature vectors and go the padded way)."""
    return hasattr(seq, "csr_item") and getattr(seq, "feature", "atomic") == "atomic"


# --------------------------------------------------------------------------- model_config of the HDF5 files
def keras_model_config(spec: ModelSpec) -> str:
    """The ``model_config`` attribute of a full-model HDF5 file (scann_model.py:165-177 saves the whole model): the
    layers of ``create_model`` (scann_model.py:329-453) in graph order with the names Keras gives them and the
    ``get_config`` dictionaries of the reference's own layers (attention.py:42-50,218-231,320-331;
    custom_layers.py:67-75).  It carries everything ``spec_from_model_config`` needs to rebuild the model without a
    yaml; it does NOT carry Keras' ``inbound_nodes`` wiring, so ``keras.models.load_model`` cannot rebuild the graph
    from a file written here (``load_weights`` on a model built by the reference's ``create_model`` can read it)."""
    import json
    L = []

    def add(cls, name, **cfg):
        L.append({"class_name": cls, "name": name, "config": dict(cfg, name=name)})

    E = spec.embedding_dim
    if spec.feature == "cgcnn":
        add("Dense", "embed_atom", units=E, activation="linear")
    else:
        add("Embedding", "embed_atom", input_dim=spec.n_atoms, output_dim=E)
    if spec.use_ring:
        add("Dense", "extra_embed", units=10, activation="linear")
    add("Dense", "dense_embed", units=spec.local_dim, activation="swish")
    add("Dropout", "dropout", rate=0.1)
    add("GaussianExpansion", "gaussian_expansion", centers=np.linspace(0, spec.gaussian_d, 20).tolist(), width=0.5)
    if spec.g_update:
        add("Dense", "neighbor_d", units=spec.local_dim, activation="swish")
        add("GaussianExpansion", "gaussian_expansion_1", centers=np.linspace(0, np.pi * 2, 20).tolist(), width=0.5)
        add("Dense", "neighbor_w", units=spec.local_dim, activation="swish")
    for l in range(spec.n_attention):
        sfx = "" if l == 0 else f"_{l}"
        add("LocalAttention", "local_attention" + sfx, dim=spec.local_dim, num_head=spec.num_head, v_proj=False, scale=0.5,
            kq_proj=True, dropout=bool(spec.use_drop), g_update=bool(spec.g_update))
        if spec.use_attn_norm:
            add("ResidualNorm", "residual_norm" + sfx, dim=spec.local_dim, dropout=0.1)
    add("Dense", "after_Lc", units=spec.local_dim, activation="swish")
    add("GlobalAttention", "global_attention", dim=spec.global_dim, v_proj=False, kq_proj=True, norm=bool(spec.use_ga_norm))
    add("Dense", "bf_property", units=spec.dense_out, activation="swish")
    add("Dense", "predict_property", units=1, activation="mrelu" if spec.mrelu_head else "linear")
    return json.dumps({"class_name": "Functional", "config": {"name": "model", "layers": L}, "backend": "tensorflow",
                       "keras_version": "2.10.0"})


def spec_from_model_config(model_config) -> ModelSpec:
    """ModelSpec from the ``model_config`` JSON of a full-model HDF5 file -- written here or by Keras 2.10 for the
    reference's graph (same layer classes, names and ``get_config`` keys): what ``load_model(path)`` gets from the file
    instead of a yaml (scann_model.py:85-96)."""
    import json
    if isinstance(model_config, bytes):
        model_config = model_config.decode()
    cfg = json.loads(model_config) if isinstance(model_config, str) else model_config
    layers = cfg["config"]["layers"]
    by_name = {l.get("name", l["config"].get("name")): l for l in layers}
    la = [l for l in layers if l["class_name"] == "LocalAttention"]
    ga = [l for l in layers if l["class_name"] == "GlobalAttention"]
    if not la or not ga or "embed_atom" not in by_name:
        raise ValueError("model_config does not describe a SCANN graph (no LocalAttention / GlobalAttention / embed_atom)")
    emb = by_name["embed_atom"]
    cgcnn = emb["class_name"] == "Dense"
    gexp = [l for l in layers if l["class_name"] == "GaussianExpansion"]
    last = by_name.get("predict_property", {"config": {}})["config"].get("activation", "linear")
    act = last if isinstance(last, str) else str(last.get("config", last))
    c0 = la[0]["config"]
    return ModelSpec(
        n_atoms=int(emb["config"].get("input_dim", 0)) if not cgcnn else 0,
        embedding_dim=int(emb["config"]["units" if cgcnn else "output_dim"]),
        n_attention=len(la), local_dim=int(c0["dim"]), num_head=int(c0["num_head"]),
        global_dim=int(ga[0]["config"]["dim"]), dense_out=int(by_name["bf_property"]["config"]["units"]),
        use_attn_norm=any(l["class_name"] == "ResidualNorm" for l in layers), use_ga_norm=bool(ga[0]["config"]["norm"]),
        use_ring="extra_embed" in by_name, g_update=bool(c0["g_update"]),
        gaussian_d=float(max(gexp[0]["config"]["centers"])) if gexp else 4.0,
        feature="cgcnn" if cgcnn else "atomic", use_drop=bool(c0.get("dropout", False)),
        target="e_b" if "mrelu" in act else "homo")


def spec_from_h5(path: str) -> ModelSpec:
    from . import h5lite
    f = h5lite.File(path)
    if "model_config" not in f.attrs:
        raise ValueError(f"{path}: no model_config attribute (a weights-only file); pass the yaml config instead")
    mc = f.attrs["model_config"]
    if isinstance(mc, np.ndarray):
        mc = mc.reshape(-1)[0] if mc.size == 1 else mc.tobytes()
    return spec_from_model_config(mc)


# --------------------------------------------------------------------------- keras-like model
class ScannKerasModel:
    """What ``SCANN.model`` exposes.  ``infer=True`` is the re-wrapped model of
    scann_model.py:79-83 whose ``predict`` returns ``[target, ga_score]``."""

    input_names = ["atomic", "atom_mask", "neighbors", "neighbor_mask", "neighbor_weight", "neighbor_distance"]

    def __init__(self, spec: ModelSpec, arena: Optional[np.ndarray] = None, infer: bool = False, seed: int = 1,
                 device: Optional[torch.device] = None, deterministic: Optional[bool] = None):
        self.spec = spec
        self.infer = infer
        # deterministic: bitwise-reproducible training (Engine); None = SCANN_DETERMINISTIC / TF_DETERMINISTIC_OPS
        self.engine = Engine(spec, arena, device=device, seed=seed, deterministic=deterministic)
        self.layout: ParamLayout = self.engine.layout
        self.lr = 1e-3
        self.allreduce = None
        self.world_size = 1
        self._y_host = None
        self.last_e2e_bytes = (0, 0)
        # Keras applies the Dropout layers (rate 0.1 after dense_embed and in every ResidualNorm,
        # scann_model.py:374, attention.py:29) whenever fit / train_on_batch run the graph with training=True
        self.dropout = True

    # ---- inference -------------------------------------------------------------------------
    def predict(self, inputs: Dict[str, object], batch_size: Optional[int] = None, verbose: int = 0,
                local_attention: bool = False):
        """Keras ``Model.predict``: numpy in, numpy out.  Keras would split the batch into
        sub-batches of 32; structures are independent so one pass gives identical results.

        ``local_attention=True`` appends the local-attention scores of every layer, one float32 array
        [n_attention, B, num_head, M, N]: ``[y, ga, la]`` in infer mode, ``[y, la]`` otherwise.  Element l is what the
        reference's layer ``local_attention[_l]`` returns as ``output[0]`` (the softmax over each atom's neighbour
        slots, scann/layers/attention.py:186-189): masked slots are 0 and an atom without valid neighbours has 1/N in
        every slot.  The other outputs are those of the plain call."""
        scores = _check_flag("local_attention", local_attention)
        eng = self.engine
        # a ragged CSR batch (DataIterator.csr_item) is expanded to the padded layout on the device
        b = eng.load_batch_csr(inputs, plan=False) if "struct_atom_off" in inputs else eng.load_batch(inputs, plan=False)
        y, ga, *la = eng.predict_step(b, replan=True, local_attention=scores)
        y_h = y.cpu().numpy().reshape(b.B, 1)          # synchronises the stream
        eng.check_status()
        self.last_e2e_bytes = (b.h2d_bytes, y.numel() * 4)
        out = [y_h]
        if self.infer:
            ga_h = ga.cpu().numpy().reshape(b.B, b.M, 1)
            self.last_e2e_bytes = (self.last_e2e_bytes[0], self.last_e2e_bytes[1] + ga.numel() * 4)
            out.append(ga_h)
        if scores:
            out.append(la[0].cpu().numpy())
            self.last_e2e_bytes = (self.last_e2e_bytes[0], self.last_e2e_bytes[1] + la[0].numel() * 4)
        return out if len(out) > 1 else y_h

    def __call__(self, inputs, training: bool = False):
        return self.predict(inputs)

    def predict_structures(self, structs, d_t: float = 4.0, w_t: float = 0.4, angle: Optional[bool] = None,
                           batch_size: int = 128, cutoff: float = 13.0, allow_pathological: bool = False,
                           local_attention: bool = False, atomic_features=None, ring_aromatic=None):
        """Structures in, ``[target [S, 1], ga_score]`` out: the README flow (``compute_voronoi_neighbor`` ->
        ``prepare_input_pmt`` -> ``predict``) for many structures, with the neighbour lists selected and batched on
        the device (``voronoi.select_neighbors``).  ``ga_score`` is a list of S float32 arrays, one value per atom,
        in input order.  The outputs equal those of ``predict`` on the same batches built on the host.

        ``angle``: the weight column, as in ``prepare_input_pmt`` (True = raw solid angle, False = normalised).  None
        picks the column ``DataIterator`` trains this model on: the raw solid angle iff ``g_update``.  (The README
        example passes ``angle=False`` to a ``g_update`` model; that feeds it a column it was not trained on.)
        ``d_t`` / ``w_t`` / ``cutoff`` / ``allow_pathological``: as in ``compute_voronoi_neighbors``.

        Batches of ``batch_size`` structures are padded to shape classes (atoms to a multiple of 8, neighbours to a
        multiple of 4 up to 32, then of 8), so that structures of different sizes replay a handful of CUDA graphs
        instead of capturing one per batch.  The padding is masked and trimmed from the outputs.

        ``feature='cgcnn'`` models need ``atomic_features``, the per-element feature table they were trained with
        ([Z + 1, 92] float32, CGCNN's ``atom_init.json`` as an array or dict): the model embeds the atomic numbers
        through it on the device (``Engine.set_atomic_features``), with the outputs of ``predict`` on the padded
        ``DataIterator(..., feature='cgcnn', atomic_features=...)`` batches of the same structures.

        ``use_ring`` models need ``ring_aromatic``: one ``[n_sites, 2]`` integer array per structure, in input order.
        These flags come from openbabel's ring and aromaticity perception, not from the geometry: pass the third item of
        the reference's ``data_energy`` rows, or run openbabel on the structures.  Each chunk's flags are uploaded once
        and copied into its batches on the device; the outputs are those of ``predict`` on the padded
        ``DataIterator(..., use_ring=True)`` batches of the same structures.

        Refused: ``use_ring`` models without ``ring_aromatic`` and ``feature='cgcnn'`` models without
        ``atomic_features`` (``NotImplementedError``); ``ring_aromatic`` for a model without ``use_ring``, flags of the
        wrong count, shape or values, structures with more than 1000 atoms (1000 is the reference's neighbour padding
        marker) or, for ``feature='cgcnn'``, with an atomic number the table has no row for (``ValueError``).

        ``local_attention=True`` returns ``[target, ga_score, la]``: ``la`` holds one ``LocalAttentionScores`` per
        structure, in input order -- every kept (site, neighbour) pair with its score in each head of each
        local-attention layer.  The scores of the padding are not copied back.  ``target`` and ``ga_score`` are those
        of the plain call."""
        from . import voronoi as V
        from .datagenerator import _refuse_ring_route, check_ring_aromatic
        scores = _check_flag("local_attention", local_attention)
        spec = self.spec
        _refuse_ring_route("predict_structures", spec.use_ring, ring_aromatic)
        if spec.feature == "cgcnn" and atomic_features is None:
            raise NotImplementedError("predict_structures: a feature='cgcnn' model embeds atoms through the per-element "
                                      "feature table it was trained with: pass atomic_features=<[Z + 1, 92] float32 "
                                      "array>")
        if spec.feature != "cgcnn" and atomic_features is not None:
            raise ValueError("predict_structures: atomic_features is the table of feature='cgcnn' models; this model "
                             "embeds atomic numbers")
        structs = list(structs)
        checked = V._arrays(structs)
        for k, X in enumerate(checked[1]):
            if len(X) == 0:
                raise ValueError(f"structure {k} has no sites")
            if len(X) > MAX_STRUCTURE_ATOMS:
                raise ValueError(f"structure {k} has {len(X)} sites: at most {MAX_STRUCTURE_ATOMS} (a neighbour index "
                                 "of 1000 is the reference's padding marker and would be masked); predict such "
                                 "structures from host-built batches: compute_voronoi_neighbors + DataIterator + predict")
        if batch_size < 1:
            raise ValueError("batch_size must be >= 1")
        column = bool(spec.g_update) if angle is None else bool(angle)
        n_at = np.array([len(X) for X in checked[1]], np.int64)
        atom_off = np.concatenate([[0], np.cumsum(n_at)])
        ring = check_ring_aromatic(ring_aromatic, n_at) if spec.use_ring else None
        eng = self.engine
        if atomic_features is not None:
            from .datagenerator import check_atomic_features, check_table_rows
            table = check_atomic_features(atomic_features)
            check_table_rows(np.concatenate([np.asarray(s.atomic_numbers).reshape(-1) for s in structs]),
                             atom_off, len(table))
            eng.set_atomic_features(table)
        y_out = np.zeros((len(structs), 1), np.float32)
        ga_out, la_out = [], []
        for c0, c1 in _structure_chunks([len(X) for X in checked[1]], batch_size):
            sel = V.select_neighbors(structs[c0:c1], d_t, w_t, column, cutoff, allow_pathological, first_index=c0,
                                     _checked=(checked[0][c0:c1], checked[1][c0:c1]))
            # the chunk's flags, uploaded once; each batch copies its contiguous atom rows on the device
            d_ring = (torch.from_numpy(ring[atom_off[c0]:atom_off[c1]]).to(sel.sel_count.device)
                      if ring is not None else None)
            for s0 in range(0, c1 - c0, batch_size):
                s1 = min(s0 + batch_size, c1 - c0)
                csr = sel.csr(s0, s1, ring=d_ring)
                M, N = shape_class(csr["M"], csr["N"])
                b = eng.load_batch_device_csr(csr, M=M, N=N, plan=False)
                y, ga, *la = eng.predict_step(b, replan=True, local_attention="csr" if scores else False)
                y_out[c0 + s0:c0 + s1, 0] = y.cpu().numpy()           # synchronises the stream
                ga_h = ga.cpu().numpy().reshape(b.B, b.M)
                ga_out.extend(ga_h[i, :n].copy() for i, n in enumerate(csr["n_atoms"]))
                if scores:
                    # the batch's pairs only, and its lists from the CSR blob on the device
                    la_out.extend(split_pair_scores(*(csr[k].cpu().numpy() for k in (
                        "struct_atom_off", "atom_nbr_off", "nbr_idx", "nbr_d")), la[0][:, :, :csr["P"]].cpu().numpy()))
        eng.check_status()
        return [y_out, ga_out, la_out] if scores else [y_out, ga_out]

    # ---- training --------------------------------------------------------------------------
    def compile(self, loss=None, optimizer=None, metrics=None, learning_rate=None):
        """``compile(loss=root_mean_squared_error, optimizer=Adam(lr, decay=1e-5), metrics=[...])``
        (scann_model.py:210-214).  The loss is fixed to RMSE + l2 terms, the optimiser to the
        Keras-2.10 Adam with decay=1e-5; ``optimizer`` / ``learning_rate`` may be a float or a schedule."""
        lr = learning_rate if learning_rate is not None else optimizer
        if lr is not None:
            self.lr = lr

    def _lr_now(self) -> float:
        return float(self.lr(self.engine.step_count)) if callable(self.lr) else float(self.lr)

    def _train_on_batch_async(self, inputs: Dict[str, object], y_true):
        """``train_on_batch`` without the blocking read: the step is queued and ``(pinned [loss, rmse, mae, _],
        event)`` is returned (Engine.loss_value_async).  ``fit`` uses it to keep one step queued behind the running
        one: the next batch's host->device copy overlaps the kernels, the losses are read at the end of the epoch
        -- Keras' fit does the same with its asynchronous metric tensors."""
        eng = self.engine
        eng.train_dropout = bool(self.dropout) and eng.use_chain and eng.use_wgrad_batch
        if isinstance(inputs, Batch):             # gathered on the device (Engine.load_batch_gather), targets included
            b, y_true = inputs, inputs.target
        elif "struct_atom_off" in inputs:
            b = eng.load_batch_csr(inputs, target=y_true, plan=False)
            y_true = b.target
        else:
            b = eng.load_batch(inputs, plan=False)
        batch_global = b.B * self.world_size
        eng.train_step(b, y_true, self._lr_now(), allreduce=self.allreduce, batch_global=batch_global, replan=True)
        self.last_e2e_bytes = (b.h2d_bytes, 16)
        return eng.loss_value_async(batch_global)

    def train_on_batch(self, inputs: Dict[str, object], y_true, return_dict: bool = False):
        """One Keras ``train_step``: returns the loss (RMSE + l2 penalties) of the batch."""
        eng = self.engine
        eng.train_dropout = bool(self.dropout) and eng.use_chain and eng.use_wgrad_batch
        if "struct_atom_off" in inputs:           # ragged CSR batch: inputs and targets in one copy, packed on device
            b = eng.load_batch_csr(inputs, target=y_true, plan=False)
            y_true = b.target
        else:
            b = eng.load_batch(inputs, plan=False)
        batch_global = b.B * self.world_size
        eng.train_step(b, y_true, self._lr_now(), allreduce=self.allreduce, batch_global=batch_global, replan=True)
        out = eng.loss_value(batch_global).cpu().numpy()       # synchronises the stream
        eng.check_status()
        self.last_e2e_bytes = (b.h2d_bytes, 16)
        if return_dict:
            return {"loss": float(out[0]), "rmse": float(out[1]), "mae": float(out[2])}
        return float(out[0])

    def evaluate_batch(self, inputs, y_true) -> Dict[str, float]:
        y = self.predict(inputs)
        return _batch_errors(y[0] if isinstance(y, list) else y, y_true)

    def _use_table_of(self, data) -> None:
        """A feature='cgcnn' model on a ``DeviceDataIterator``: embed through the iterator's feature table."""
        if self.spec.feature == "cgcnn" and getattr(data, "atomic_features", None) is not None:
            self.engine.set_atomic_features(data.atomic_features)

    def predict_device_batch(self, data, idx: int):
        """Predictions of batch ``idx`` of a ``DeviceDataIterator``, gathered on the device: ``(y [B, 1], targets
        [B])`` as host float32 arrays -- the same values ``predict(data[idx][0])`` gives."""
        eng = self.engine
        self._use_table_of(data)
        b = eng.load_batch_gather(data, *data.batch_shape(idx), plan=False)
        y, _ = eng.predict_step(b, replan=True)
        y_h = y.cpu().numpy().reshape(b.B, 1)          # synchronises the stream
        self.last_e2e_bytes = (0, y.numel() * 4)
        return y_h, data.batch_target(idx)

    def fit(self, x, epochs: int = 1, validation_data=None, callbacks=None, verbose: int = 2, shuffle: bool = False,
            **_ignored) -> History:
        """``model.fit(trainIter, epochs, validation_data=validIter, ...)`` (scann_model.py:232-241) over a
        ``Sequence``-like iterator (``len``, ``__getitem__`` -> (inputs, target), ``on_epoch_end``).  A
        ``DeviceDataIterator`` (as ``x`` or as ``validation_data``) has its batches gathered on the device."""
        from .datagenerator import DeviceDataIterator
        on_device = isinstance(x, DeviceDataIterator)
        hist = History()
        callbacks = list(callbacks or [])
        self.stop_training = False
        for cb in callbacks:                      # Keras callback protocol (scann_b200/callbacks.py)
            if hasattr(cb, "set_model"):
                cb.set_model(self)
            if hasattr(cb, "on_train_begin"):
                cb.on_train_begin({})
        for ep in range(epochs):
            for cb in callbacks:
                if hasattr(cb, "on_epoch_begin"):
                    cb.on_epoch_begin(ep, {})
            losses, maes, pending = [], [], []

            def harvest(upto: int) -> None:
                while len(pending) > upto:
                    pin, ev = pending.pop(0)
                    ev.synchronize()
                    losses.append(float(pin[0]))
                    maes.append(float(pin[2]))

            eng = self.engine
            if on_device:
                self._use_table_of(x)
            eng.overlap_h2d = True
            try:
                for i in range(len(x)):
                    if on_device:                 # a device-resident data set: no host->device copy at all
                        inputs, target = eng.load_batch_gather(x, *x.batch_shape(i), plan=False), None
                    else:
                        # iterators that can hand out the ragged CSR form skip the host-side padding altogether
                        inputs, target = x.csr_item(i) if _ragged_capable(x) else x[i]
                    pending.append(self._train_on_batch_async(inputs, target))
                    harvest(4)                    # results older than 4 steps (long finished; ring of 8 slots)
                harvest(0)
            finally:
                eng.overlap_h2d = False
            eng.check_status()
            hist.add("loss", float(np.mean(losses)))
            hist.add("mae", float(np.mean(maes)))
            if validation_data is not None:
                if isinstance(validation_data, DeviceDataIterator):
                    v = [_batch_errors(*self.predict_device_batch(validation_data, i))
                         for i in range(len(validation_data))]
                    eng.check_status()
                else:
                    v = [self.evaluate_batch(*validation_data[i]) for i in range(len(validation_data))]
                hist.add("val_mae", float(np.mean([m["mae"] for m in v])))
            if hasattr(x, "on_epoch_end"):
                x.on_epoch_end()
            if verbose:
                print(f"Epoch {ep + 1}/{epochs} - " + " - ".join(f"{k}: {vals[-1]:.6f}" for k, vals in hist.history.items()))
            logs = {k: vals[-1] for k, vals in hist.history.items()}
            for cb in callbacks:
                if hasattr(cb, "on_epoch_end"):
                    cb.on_epoch_end(ep, logs)
            if self.stop_training:
                break
        for cb in callbacks:
            if hasattr(cb, "on_train_end"):
                cb.on_train_end({})
        return hist

    # ---- weights ---------------------------------------------------------------------------
    def get_weights(self):
        """Weights in the reference's Keras order (see params.ParamLayout)."""
        d = self.layout.to_dict(self.engine.get_params())
        return [d[e.name].copy() for e in self.layout]

    def set_weights(self, weights: Iterable[np.ndarray]) -> None:
        weights = list(weights)
        if len(weights) != len(self.layout.entries):
            raise ValueError(f"expected {len(self.layout.entries)} arrays, got {len(weights)}")
        self.engine.set_params(self.layout.from_dict({e.name: w for e, w in zip(self.layout, weights)}))

    # ---- weights: Keras legacy HDF5 (.h5, what the reference's model.save / ModelCheckpoint / load_model use,
    #      scann_model.py:79-96,223-230) or .npz with the same names -------------------------------------------
    def _keras_layers(self):
        """[(layer name, [(weight name ":0", array)])] in ParamLayout (= Keras layer / weight) order."""
        d = self.layout.to_dict(self.engine.get_params())
        layers, index = [], {}
        for e in self.layout:
            lname = e.name.split("/")[0]
            if lname not in index:
                index[lname] = len(layers)
                layers.append((lname, []))
            layers[index[lname]][1].append((e.name + ":0", d[e.name]))
        return layers

    def save_weights(self, path: str) -> None:
        if path.endswith((".h5", ".hdf5", ".keras")):
            from . import h5lite
            h5lite.save_keras_weights(path, self._keras_layers(), full_model=False)
            return
        d = self.layout.to_dict(self.engine.get_params())
        np.savez(path, **{k.replace("/", "__"): v for k, v in d.items()})

    def save(self, path: str) -> None:
        """``model.save("...h5")``: full-model layout (weights under /model_weights)."""
        if path.endswith((".h5", ".hdf5", ".keras")):
            from . import h5lite
            h5lite.save_keras_weights(path, self._keras_layers(), full_model=True, model_config=keras_model_config(self.spec))
        else:
            self.save_weights(path)

    def load_weights(self, path: str) -> None:
        if path.endswith((".h5", ".hdf5", ".keras")):
            self.engine.set_params(self.layout.from_dict(self._from_keras_h5(path)))
            return
        with np.load(path) as z:
            d = {k.replace("__", "/"): z[k] for k in z.files}
        self.engine.set_params(self.layout.from_dict(d))

    def _from_keras_h5(self, path: str) -> Dict[str, np.ndarray]:
        """Maps a Keras-2.10 HDF5 file onto the parameter layout the way ``keras.Model.load_weights`` does:
        layers are matched by name (the top-level layer names of create_model are explicit or Keras' automatic
        ``local_attention_<i>`` / ``residual_norm_<i>``), the weights of a layer by ORDER (= creation order of the
        layer's variables), with every shape checked; layers without weights (Input, Lambda, Dropout, ...) are
        skipped."""
        from . import h5lite
        per_layer = {}
        for e in self.layout:
            per_layer.setdefault(e.name.split("/")[0], []).append(e)
        out, seen = {}, set()
        file_layers = [(n, ws) for n, ws in h5lite.load_keras_weights(path) if ws]
        if any(n not in per_layer for n, _ in file_layers):
            # Keras' automatic names carry a per-session counter (a model built second in a session is saved with
            # local_attention_7 ...): fall back to what keras load_weights itself does for topological loading --
            # the weight-bearing layers IN ORDER, shapes checked below
            if len(file_layers) != len(per_layer):
                raise ValueError(f"{path}: {len(file_layers)} layers with weights, the model expects {len(per_layer)}")
            file_layers = [(mine, ws) for (_, ws), mine in zip(file_layers, per_layer)]
        for lname, ws in file_layers:
            if lname not in per_layer:
                raise ValueError(f"{path}: layer {lname!r} with weights is not part of this model configuration")
            ents = per_layer[lname]
            if len(ws) != len(ents):
                raise ValueError(f"{path}: layer {lname!r} has {len(ws)} weights, the model expects {len(ents)}")
            for (wname, arr), e in zip(ws, ents):
                if tuple(arr.shape) != e.shape:
                    raise ValueError(f"{path}: {lname}/{wname} has shape {tuple(arr.shape)}, expected {e.shape} ({e.name})")
                out[e.name] = np.asarray(arr, np.float32)
            seen.add(lname)
        missing = [l for l in per_layer if l not in seen]
        if missing:
            raise ValueError(f"{path}: no weights for layers {missing}")
        return out

    def count_params(self) -> int:
        return self.layout.n_params

    def summary(self) -> None:
        print(f"Model: SCANN ({'SCANN+' if self.spec.g_update else 'SCANN'}), {self.spec.n_attention} local-attention layers")
        for e in self.layout:
            print(f"  {e.name:50s} {str(e.shape):14s} {e.size}")
        print(f"Total params: {self.layout.n_params}")

    def get_layer(self, name: str):
        if name != "global_attention":
            raise ValueError(f"No such layer: {name}")
        return self


def create_model(config: dict, seed: int = 1, infer: bool = False, arena: Optional[np.ndarray] = None,
                 deterministic: Optional[bool] = None) -> ScannKerasModel:
    """Counterpart of ``create_model(config)`` (scann_model.py:329-453).  ``deterministic``: see ``Engine``."""
    return ScannKerasModel(model_spec(config), arena=arena, infer=infer, seed=seed, deterministic=deterministic)


class SCANN:
    """Same constructor and methods as the reference facade (scann_model.py:42-96, 315-319)."""

    def __init__(self, config=None, pretrained: str = "", mode: str = "train"):
        self.config = config
        self.model = None
        self.mean, self.std = 0, 1
        if "target_mean" in self.config["hyper"]:                       # scann_model.py:66-68
            self.mean = float(self.config["hyper"]["target_mean"])
            self.std = float(self.config["hyper"]["target_std"])
        if mode in ("train", "eval"):                                   # :70-77
            self.model = create_model(self.config)
            if pretrained:
                print("load pretrained model from ", pretrained, "\n")
                self.model.load_weights(pretrained)
                self.config["hyper"]["pretrained"] = pretrained
        else:                                                           # :78-83
            if not pretrained:
                raise ValueError("mode='infer' needs pretrained weights (the reference calls load_model(pretrained))")
            self.model = create_model(self.config, infer=True)
            self.model.load_weights(pretrained)

    @classmethod
    def load_model_infer(cls, path: str, config: Optional[dict] = None):
        """``SCANN.load_model_infer(path)`` (scann_model.py:85-91): the graph comes from the file's ``model_config``
        (``config`` = a yaml dict is optional, for weights-only files)."""
        m = (create_model(config, infer=True) if config is not None
             else ScannKerasModel(spec_from_h5(path), infer=True))
        m.load_weights(path)
        return m

    @classmethod
    def load_model(cls, path: str, config: Optional[dict] = None):
        """``SCANN.load_model(path)`` (scann_model.py:93-96)."""
        m = create_model(config) if config is not None else ScannKerasModel(spec_from_h5(path))
        m.load_weights(path)
        return m

    def predict_data(self, ip):                                         # :315-319
        out = self.model.predict(ip)
        if len(out) == 2:
            return out[0] * self.std + self.mean, out[1]
        return out * self.std + self.mean

    def _predict_structures(self, structs, d_t: float = 4.0, w_t: float = 0.4, angle: Optional[bool] = None,
                            batch_size: int = 128, cutoff: float = 13.0, allow_pathological: bool = False,
                            local_attention: bool = False, atomic_features=None, ring_aromatic=None):
        """``ScannKerasModel.predict_structures`` with the target scaled back like ``predict_data``."""
        y, *rest = self.model.predict_structures(structs, d_t=d_t, w_t=w_t, angle=angle, batch_size=batch_size,
                                                 cutoff=cutoff, allow_pathological=allow_pathological,
                                                 local_attention=local_attention, atomic_features=atomic_features,
                                                 ring_aromatic=ring_aromatic)
        return (y * self.std + self.mean, *rest)

    @property
    def predict_structures(self):
        """``predict_structures(structs, d_t=4.0, w_t=0.4, angle=None, batch_size=128, cutoff=13.0,
        allow_pathological=False, local_attention=False, atomic_features=None, ring_aromatic=None)``:
        ``ScannKerasModel.predict_structures`` with the target scaled back like ``predict_data``.  (A property, not a
        plain method: the record of SCANN's plain public methods in tests/golden/reference/graph_public_surface.npz stays
        the surface that was compared with the reference's SCANN, which has no such method.)"""
        return functools.partial(SCANN._predict_structures, self)

    # ---- training shell (scann_model.py:163-313) ------------------------------------------------------------
    def _run_dir(self) -> str:
        hy = self.config["hyper"]
        return "{}_{}".format(hy["save_path"], hy["target"])

    def prepare_dataset(self, split: bool = True):
        """``SCANN.prepare_dataset`` (scann_model.py:98-161): load the pickled data set (``hyper.data_energy_path`` /
        ``hyper.data_nei_path``, written by the reference's preprocessing), standardise the target when
        ``hyper.scaler`` is set (float32 mean / std, recorded in the config as strings like the reference), split it
        with the global numpy generator and attach ``trainIter`` / ``validIter`` / ``testIter`` (or ``dataIter``)."""
        from .datagenerator import DataIterator, load_dataset
        hy, cm = self.config["hyper"], self.config["model"]
        data_energy, data_neighbor = load_dataset(hy["data_energy_path"], hy["data_nei_path"], hy["target"],
                                                  use_ref=hy["use_ref"], use_ring=cm["use_ring"])
        self._scale_targets(data_energy)

        def iterator(indices=None, shuffle=False):
            return DataIterator(batch_size=hy["batch_size"], use_ring=cm["use_ring"], shuffle=shuffle,
                                feature=cm["feature"], g_update=cm["g_update"],
                                data_neighbor=data_neighbor if indices is None else data_neighbor[indices],
                                data_energy=data_energy if indices is None else data_energy[indices])

        return self._attach_iterators(len(data_energy), iterator, split)

    def _scale_targets(self, data_energy) -> None:
        """Standardise column 1 of the rows in place when ``hyper.scaler`` is set (float32 mean / std) and record the
        scaling and the data-set size in the config (scann_model.py:117-131)."""
        hy = self.config["hyper"]
        if hy["scaler"]:
            values = [row[1] for row in data_energy]
            self.mean, self.std = np.mean(values, dtype="float32"), np.std(values, dtype="float32")
            print("Normalize dataset property with mean: ", self.mean, " , std: ", self.std, "\n")
            data_energy[:, 1] = (data_energy[:, 1] - self.mean) / self.std
        hy["target_mean"], hy["target_std"] = str(self.mean), str(self.std)
        hy["data_size"] = len(data_energy)

    def _attach_iterators(self, n: int, iterator, split: bool):
        """``dataIter``, or the train | valid | test split of the global numpy generator (scann_model.py:133-161)."""
        from .datagenerator import split_data
        hy = self.config["hyper"]
        if not split:
            self.dataIter = iterator()
            return None
        train, valid, test, extra = split_data(len_data=n, test_percent=hy["test_percent"],
                                               train_size=hy["train_size"], test_size=hy["test_size"])
        assert len(extra) == 0, "Split was inexact {} {} {} {}".format(len(train), len(valid), len(test), len(extra))
        print("Number of train data : ", len(train), " , Number of valid data: ", len(valid),
              " , Number of test data: ", len(test), "\n")
        # the reference shuffles every subset that is as long as the training subset (scann_model.py:146)
        self.trainIter, self.validIter, self.testIter = [iterator(ix, shuffle=(len(ix) == len(train)))
                                                         for ix in (train, valid, test)]
        return train, valid, test

    def _prepare_structures(self, structs, targets, split: bool = True, atomic_features=None, ring_aromatic=None,
                            **voronoi_args):
        """``SCANN.prepare_structures``: see the property."""
        from .datagenerator import DeviceDataIterator, _refuse_structures_route, check_ring_aromatic
        hy, cm = self.config["hyper"], self.config["model"]
        _refuse_structures_route("SCANN.prepare_structures", cm["use_ring"], cm["feature"], atomic_features,
                                 ring_aromatic)
        structs = list(structs)
        targets = list(np.asarray(targets, dtype=object).reshape(-1))
        if len(targets) != len(structs):
            raise ValueError(f"{len(structs)} structures but {len(targets)} targets")
        ring = None
        if cm["use_ring"]:              # checked in the caller's order, so that an error names the caller's index
            n_at = [len(np.asarray(s.cart_coords).reshape(-1, 3)) for s in structs]
            atom_off = np.concatenate([[0], np.cumsum(n_at, dtype=np.int64)])
            flat = check_ring_aromatic(ring_aromatic, n_at)
            ring = [flat[atom_off[k]:atom_off[k + 1]] for k in range(len(structs))]
        rows = np.empty((len(structs), 2), dtype=object)          # the rows of load_dataset: [atoms, target]
        rows[:, 1] = [float(t) for t in targets]
        self._scale_targets(rows)

        def iterator(indices=None, shuffle=False):
            ix = range(len(structs)) if indices is None else indices
            return DeviceDataIterator.from_structures([structs[k] for k in ix], rows[list(ix), 1],
                                                      batch_size=hy["batch_size"], shuffle=shuffle,
                                                      g_update=cm["g_update"], use_ring=cm["use_ring"],
                                                      feature=cm["feature"],
                                                      atomic_features=atomic_features if cm["feature"] == "cgcnn" else None,
                                                      ring_aromatic=[ring[k] for k in ix] if ring is not None else None,
                                                      **voronoi_args)

        return self._attach_iterators(len(structs), iterator, split)

    @property
    def prepare_structures(self):
        """``prepare_structures(structs, targets, split=True, atomic_features=None, ring_aromatic=None,
        **voronoi_args)``: ``prepare_dataset`` for structures and their targets instead of the reference's data files.
        The same target scaling (``hyper.scaler``), config entries and split of the global numpy generator;
        ``trainIter`` / ``validIter`` / ``testIter`` (or ``dataIter``) are ``DeviceDataIterator.from_structures``
        (``voronoi_args``: ``d_t``, ``w_t``, ``angle``, ``cutoff``, ``allow_pathological``, ``converter``), so training
        and evaluation gather their batches on the device.  ``feature='cgcnn'`` models need ``atomic_features``, their
        per-element feature table ([Z + 1, 92] float32).  ``use_ring`` models (``model.use_ring`` of the config) need
        ``ring_aromatic``, one ``[n_sites, 2]`` integer array per structure (the third item of the reference's
        ``data_energy`` rows, or openbabel's perception run on the structures); the flags follow their structures
        through the split, as ``prepare_dataset``'s rows do.  Refused for ``use_ring`` models without ``ring_aromatic``
        and for ``feature='cgcnn'`` without ``atomic_features``.  (A property for the same reason as
        ``predict_structures``.)"""
        return functools.partial(SCANN._prepare_structures, self)

    def create_callbacks(self):
        """ModelCheckpoint(best val_mae) + EarlyStopping(patience 200) + SGDRC / lr logging (scann_model.py:163-197)."""
        from . import callbacks as C
        hy = self.config["hyper"]
        cbs = [C.ModelCheckpoint(filepath="{}/models/model_{}.h5".format(self._run_dir(), hy["target"]), monitor="val_mae",
                                 save_weights_only=False, verbose=2, save_best_only=True),
               C.EarlyStopping(monitor="val_mae", patience=200)]
        if hy.get("scheduler") == "sgdr":
            lr = C.SGDRC(lr_min=hy["min_lr"], lr_max=hy["lr"], t0=50, tmult=2, lr_max_compression=1.2, trigger_val_mae=300)
            cbs += [lr, C.LearningRateScheduler(lr.lr_scheduler)]
        else:
            cbs.append(C.LearningRateLoggingCallback())
        return cbs

    def train(self, epochs: int = 1000):
        """``SCANN.train`` (scann_model.py:199-245) for iterators attached as ``self.trainIter`` / ``self.validIter``
        or by ``prepare_dataset``)."""
        import yaml
        if not hasattr(self, "trainIter"):
            raise RuntimeError("attach trainIter / validIter (DataIterator-like sequences) before train()")
        os.makedirs(os.path.join(self._run_dir(), "models"), exist_ok=True)
        with open(os.path.join(self._run_dir(), "config.yaml"), "w") as f:
            yaml.safe_dump(self.config, f, default_flow_style=False)
        self.train_iterators(self.trainIter, getattr(self, "validIter", None), epochs, self.create_callbacks())
        # the reference deletes the trained model here (scann_model.py:243-245), so that evaluate() runs on the best
        # val_mae checkpoint, not on the last epoch's weights; the engine object is kept, its weights are reloaded
        self._evaluate_from_checkpoint = True

    def evaluate(self):
        """``SCANN.evaluate`` (scann_model.py:247-313): best checkpoint -> test predictions -> R2 / MAE report."""
        hy = self.config["hyper"]
        best = "{}/models/model_{}.h5".format(self._run_dir(), hy["target"])
        if self.model is None or (getattr(self, "_evaluate_from_checkpoint", False) and os.path.exists(best)):
            print("Load best validation weight for predicting testset", "\n")
            if self.model is None:
                self.model = create_model(self.config)
            self.model.load_weights(best)
            self._evaluate_from_checkpoint = False
        from .datagenerator import DeviceDataIterator
        data = self.dataIter if hasattr(self, "dataIter") else self.testIter
        y, y_predict = [], []
        for i in range(len(data)):
            if isinstance(data, DeviceDataIterator):
                out, target = self.model.predict_device_batch(data, i)
            else:
                inputs, target = data[i]
                out = self.model.predict(inputs)
                out = out[0] if isinstance(out, list) else out
            y.extend(np.asarray(target, np.float64).reshape(-1).tolist())
            y_predict.extend(np.asarray(out, np.float64).reshape(-1).tolist())
            if i % 10 == 0:
                print(f"{i}/{len(data)}")
        if isinstance(data, DeviceDataIterator):
            self.model.engine.check_status()
        ya, yp = np.asarray(y), np.asarray(y_predict)
        mae = float(np.abs(ya - yp).mean()) * self.std
        ss_tot = float(((ya - ya.mean()) ** 2).sum())
        r2 = 1.0 - float(((ya - yp) ** 2).sum()) / ss_tot if ss_tot > 0 else 0.0     # sklearn.metrics.r2_score
        print("Result for testset ", hy["target"], " : R2 score: ", r2, " and MAE: ", mae)
        os.makedirs(self._run_dir(), exist_ok=True)
        lines = []
        if hasattr(self, "hist"):
            np.save(os.path.join(self._run_dir(), "hist_data.npy"),
                    np.array([y_predict, y, self.hist.history], dtype=object), allow_pickle=True)
            lines.append("Training MAE: " + str(min(self.hist.history["mae"]) * self.std) + "\n")
            if "val_mae" in self.hist.history:
                lines.append("Val MAE: " + str(min(self.hist.history["val_mae"]) * self.std) + "\n")
        lines.append("Test MAE: " + str(mae) + ", Test R2: " + str(r2))
        with open(os.path.join(self._run_dir(), "report.txt"), "w") as f:
            f.writelines(lines)
        return {"mae": mae, "r2": r2}

    def train_iterators(self, train_iter, valid_iter=None, epochs: int = 1000, callbacks=None):
        """``train`` (scann_model.py:199-241) minus dataset loading: lr schedule + compile + fit."""
        hy = self.config["hyper"]
        if hy.get("scheduler") == "sgdr":
            lr = hy["lr"]
        else:
            lr = CosineDecay(hy["lr"], 0.5 * len(train_iter) * epochs, alpha=hy["min_lr"] / hy["lr"])
        self.model.compile(optimizer=lr)
        self.hist = self.model.fit(train_iter, epochs=epochs, validation_data=valid_iter, callbacks=callbacks)
        return self.hist
