"""Device engine: orchestrates the sm_100a kernels for one SCANN model on one GPU.

Host logic only (Python): owns the flat parameter / gradient arenas and the per-shape
workspaces, and issues the C-ABI kernel calls on the current torch CUDA stream.  torch is
used for device memory, streams and host<->device copies -- never for arithmetic on the
hot path.  Graph being executed: ``create_model`` of the reference
(scann/models/scann_model.py:329-453); see DESIGN.md for the kernel schedule.
"""
from __future__ import annotations

import ctypes
import os
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _abi
from ._abi import ChainStep, WgradProblem, chain_step, check, lib, ptr_array
from .config import ModelSpec, N_RBF, check_kernel_support
from .dlpack import import_tensor
from .params import ParamLayout, layer_name

TILE = 128
PLAN_GSZ = 128
TABLE_ROUTE = "atomic_features"     # last item of the graph keys of cgcnn batches embedded through the table
D = 128
L2_COEF = 1e-4

ERR_BITS = {1: "plan tile capacity exceeded", 2: "an atom has more than 128 valid neighbours",
            4: "atomic number outside the embedding table", 8: "neighbour index outside [0, M)",
            16: "a bounded mbarrier wait of a pipelined kernel (local attention, chained Dense) gave up"}


def deterministic_mode(deterministic: Optional[bool] = None, environ=None) -> bool:
    """Whether an engine trains in the deterministic mode (DESIGN.md section 4.7).  An explicit ``deterministic``
    wins; None reads the environment: ``SCANN_DETERMINISTIC=1``, or the reference's own switch
    ``TF_DETERMINISTIC_OPS`` set to ``1`` / ``true`` (the reference's train.py:16-25 sets it)."""
    if deterministic is not None:
        return bool(deterministic)
    env = os.environ if environ is None else environ
    return (env.get("SCANN_DETERMINISTIC", "0") == "1"
            or env.get("TF_DETERMINISTIC_OPS", "").strip().lower() in ("1", "true"))


def _p(t: Optional[torch.Tensor], off_elems: int = 0) -> int:
    if t is None:
        return 0
    return t.data_ptr() + off_elems * t.element_size()


class Batch:
    """Device-resident inputs of one padded batch plus its pair plan."""

    def __init__(self):
        self.B = self.M = self.N = self.R = 0
        self.tile_cap = 0
        self.P_host = None          # number of valid pairs when known on the host
        self.A_host = None
        # feature='cgcnn' only: TABLE_ROUTE when the batch carries atomic numbers (CSR / gathered batches, embedded
        # through the engine's per-element table), None when it carries the padded feature vectors (load_batch)
        self.route = None


class Engine:
    def __init__(self, spec: ModelSpec, arena: Optional[np.ndarray] = None, device: Optional[torch.device] = None,
                 seed: int = 1, deterministic: Optional[bool] = None):
        """``deterministic``: bitwise-reproducible train steps (DESIGN.md section 4.7); None reads the environment
        (``deterministic_mode``).  Fixed for the life of the engine."""
        check_kernel_support(spec)
        self.deterministic = deterministic_mode(deterministic)
        self.sm_count = _abi.require_gpu()
        self.device = device or torch.device("cuda", torch.cuda.current_device())
        self.spec = spec
        self.layout = ParamLayout(spec)
        n = self.layout.total
        if arena is None:
            arena = self.layout.init_arena(seed)
        assert arena.shape == (n,)
        dev = self.device
        self.params = torch.from_numpy(np.ascontiguousarray(arena, np.float32)).to(dev)
        self.paramsT = torch.zeros(n, dtype=torch.float32, device=dev)
        # gradient arena: [0,n) gradients, [n] SSE, [n+1] sum |err|  (one all-reduce covers all)
        self.grads = torch.zeros(n + 4, dtype=torch.float32, device=dev)
        self.adam_m = torch.zeros(n, dtype=torch.float32, device=dev)
        self.adam_v = torch.zeros(n, dtype=torch.float32, device=dev)
        self.l2mask = torch.from_numpy(self.layout.l2_mask()).to(dev)
        self.grad_out = torch.zeros(n, dtype=torch.float32, device=dev)
        # word 0: flag bits (ERR_BITS); words 1..4: {wait site, CTA, tile, stage} of a pipelined kernel that gave up
        self.status = torch.zeros(8, dtype=torch.int32, device=dev)
        self.loss_out = torch.zeros(4, dtype=torch.float32, device=dev)
        # [0..7] optimiser scalars, [8..11] dropout control block (ScannDropCtl: seed, threshold, scale bits, enabled)
        self.adam_scalars = torch.zeros(16, dtype=torch.float32, device=dev)
        self._adam_host = torch.zeros(16, dtype=torch.float32).pin_memory()
        # training-mode Dropout (rate 0.1 after dense_embed and in every ResidualNorm): Keras applies it inside
        # fit(); the facade switches it on for fit / train_on_batch, direct engine users opt in
        self.train_dropout = os.environ.get("SCANN_DROPOUT", "0") == "1"
        self.dropout_rate = 0.1
        self.dropout_seed = seed
        self.last_drop_seed = 0
        self._adam_ev = None
        self.step_count = 0
        self.p2p = None        # dist.P2PExchange: gradient exchange over peer memory, fused into the optimiser kernel
        # RBF centres: np.linspace(0, gaussian_d, 20) / np.linspace(0, 2*pi, 20), float32 (scann_model.py:378,384)
        self.centers_d = torch.from_numpy(np.linspace(0, spec.gaussian_d, N_RBF, dtype="float32")).to(dev)
        self.centers_w = torch.from_numpy(np.linspace(0, np.pi * 2, N_RBF, dtype="float32")).to(dev)
        # list of 128x128 weight blocks whose transpose the backward pass needs
        offs = []
        for e in self.layout:
            if e.name.endswith("/kernel") and len(e.shape) == 2 and e.shape[1] == D and e.shape[0] % D == 0:
                for blk in range(e.shape[0] // D):
                    offs.append(e.offset + blk * D * D)
        self.tblocks = torch.tensor(offs, dtype=torch.int32, device=dev)
        import collections
        self._ws: Dict[Tuple, dict] = {}
        self._pinned: Dict[Tuple, list] = {}
        self._batches: "collections.OrderedDict[Tuple, Batch]" = collections.OrderedDict()
        # persistent device buffers + captured graphs are kept for this many batch shape classes (LRU)
        self.max_shape_classes = int(os.environ.get("SCANN_MAX_SHAPE_CLASSES", "8"))
        self.use_graphs = os.environ.get("SCANN_GRAPHS", "1") == "1"
        self.la_grid = self.sm_count
        self.launches = 0
        # shape classes dropped from the LRU above, CUDA graphs captured (train and inference)
        self.shape_class_evictions = 0
        self.graph_captures = 0
        self.prof: Optional[dict] = None
        # engine selection (tensor-core kernels are the default; SCANN_ENGINE=simt keeps the fp32 SIMT path)
        eng = os.environ.get("SCANN_ENGINE", "tc")
        self.tc_dense = eng != "simt" and os.environ.get("SCANN_DENSE", "tc") == "tc"
        self.tc_la_fwd = eng != "simt" and os.environ.get("SCANN_LA_FWD", "tc") == "tc"
        self.tc_la_bwd = self.tc_la_fwd and os.environ.get("SCANN_LA_BWD", "tc") == "tc"
        self.use_side_stream = os.environ.get("SCANN_SIDE_STREAM", "1") == "1"
        # geometry-initialisation backward beside the embedding backward at the end of the step (_backward_tail)
        self.tail_fork = os.environ.get("SCANN_TAIL_FORK", "1") == "1"
        # Wave-balanced tiles: rows per tile chosen so that the tile count is a whole number of rounds over the
        # SMs' warp groups (QM9/128: 592 tiles of ~40 rows instead of 388 of 64: every group runs two short
        # tiles instead of some running two long ones).  Local-attention backward 74 -> 64 us per layer; the
        # weight-gradient launch runs over the compact list of valid rows, so it does not pay for the padding.
        self.balance_tiles = os.environ.get("SCANN_BALANCE_TILES", "1") == "1"
        # rows per tile slot of the pair plan: 64 = two warp groups per CTA in the tensor-core local-attention
        # kernels (needs <= 64 neighbours per atom), 128 = one tile stream per CTA (also the SIMT engine)
        # 32 = the pipelined kernels (<= 32 neighbours per atom).  Default (0): 32 where the pipelined kernels apply,
        # else 64, else 128.
        self.tile_stride_pref = int(os.environ.get("SCANN_TILE_STRIDE", "0"))
        # warp-specialised TMA pipelines for the local-attention kernels (la_pipe.cu, la_pipe_bwd.cu) on plans with
        # 32-row tile slots: bit 0 geometry forward, 1 attention forward, 2 attention backward, 3 geometry backward.
        # 0 keeps the round-1 kernels (four 4-warp groups per CTA on the same 32-row plan when SCANN_TILE_STRIDE=32).
        self.la_pipe_built = 15
        self.la_pipe = (int(os.environ.get("SCANN_LA_PIPE", str(self.la_pipe_built))) & self.la_pipe_built
                        if (self.tc_la_fwd and self.tc_la_bwd) else 0)
        # g_update = False layers (model_ptgp.yaml) on the pipelined ATTENTION kernels: their geometry operand
        # g' = swish(rbf(d) Wf + bf) * w is written out per layer by scann_noupdate_geom_forward (training saves it anyway)
        # and read through TMA like the updated geometry of a g_update = True layer.  Needs both attention bits of la_pipe.
        self.noup_pipe = os.environ.get("SCANN_NOUP_PIPE", "1") == "1" and (self.la_pipe & 6) == 6
        self.side_stream = torch.cuda.Stream(device=self.device)
        self._prep_event = None
        # local-attention kernels with four warp groups per CTA where the plan's tiles hold <= 48 rows (bit mask:
        # 1 geometry forward, 2 attention forward, 4 attention backward, 8 geometry backward)
        # CTAs per SM of the SIMT geometry-initialisation kernels (latency-bound FMA chains: more resident warps)
        self.gi_fwd_mult = int(os.environ.get("SCANN_GI_FWD", "3"))
        self.gi_bwd_mult = int(os.environ.get("SCANN_GI_BWD", "2"))
        self.la_groups4 = int(os.environ.get("SCANN_LA4", "17"))      # geometry forward, staggered start
        lib.scann_set_la_groups4(self.la_groups4)
        # pipelined input feed (facade fit): a step's host->device copy runs on its own stream into a staging
        # blob while the previous step computes; the main stream only does a device-to-device hand-over
        self.overlap_h2d = False
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self._loss_ring: list = []
        # programmatic dependent launch along the forward / backward kernel chain (include/scann_b200.h)
        self.use_pdl = os.environ.get("SCANN_PDL", "1") == "1"
        # development aid: kernels to leave out of the step (results are then meaningless; only the timing
        # difference to the full step is of interest) -- comma list of wgrad,la_fwd,la_bwd,rn,geom_init
        self._skip = set(filter(None, os.environ.get("SCANN_DEBUG_SKIP", "").split(",")))
        # per-atom Dense layers between two local-attention layers fused into one chained kernel
        self.use_chain = os.environ.get("SCANN_CHAIN", "1") == "1" and self.tc_dense and self.tc_la_fwd
        # warp-specialised chained kernel (chain2_tc.cu): weight blocks as ready-made tcgen05 operand images, rebuilt
        # after every optimiser step / set_params and streamed into shared memory with cp.async.bulk
        self.use_chain2 = os.environ.get("SCANN_CHAIN2", "1") == "1" and self.use_chain
        # up to this many rows (default: one wave of 64-row tiles) the warp-specialised form runs, above it the round-1 kernel
        self.chain2_max_rows = (int(os.environ.get("SCANN_CHAIN2_MAX_ROWS", "0")) or lib.scann_dense_chain2_max_rows()) \
            if self.use_chain2 else 0
        self._wimg_index = {int(o): i for i, o in enumerate(offs)}
        self._wimg_buf = torch.empty(len(offs) * 2 * 32768 + 256, dtype=torch.float32, device=dev) if self.use_chain2 else None
        self._wimg_base = ((self._wimg_buf.data_ptr() + 1023) // 1024 * 1024) if self.use_chain2 else 0
        self._wimg_dirty = True
        # every weight-gradient GEMM of the step in one persistent launch at the end of the backward pass
        self.use_wgrad_batch = os.environ.get("SCANN_WGRAD_BATCH", "1") == "1" and self.use_chain and self.tc_la_bwd
        self._nccl_warned = False
        # feature='cgcnn': per-element feature table [Z_rows, 92] on the device (set_atomic_features), its host copy and
        # the buffers of the table route: emb_table / d_emb [Z_rows, E], G [Z_rows + 3, 128]
        self.atomic_features: Optional[torch.Tensor] = None
        self._afeat_host: Optional[np.ndarray] = None
        self._tab: Dict[str, torch.Tensor] = {}

    # ------------------------------------------------------------------ feature='cgcnn' on atomic numbers
    def set_atomic_features(self, table) -> None:
        """The per-element feature table ([Z_rows, 92] float32, row 0 = padding atom) a ``feature='cgcnn'`` model embeds
        batches that carry atomic numbers with (``load_batch_csr``, ``load_batch_device_csr``, ``load_batch_gather``):
        embed_atom's output for an atom is row Z of ``table @ W + b``, computed once per forward.  A table of the same
        shape is copied into the same device buffer in stream order (captured graphs stay valid); one with another row
        count replaces the buffer and drops the captured graphs of that route."""
        from .datagenerator import check_atomic_features
        if self.spec.feature != "cgcnn":
            raise ValueError("set_atomic_features: only feature='cgcnn' models read a per-element feature table")
        t = check_atomic_features(table)
        old = self._afeat_host
        if old is not None and old.shape == t.shape:
            if not np.array_equal(old.view(np.uint32), t.view(np.uint32)):
                self.atomic_features.copy_(torch.from_numpy(t))
                self._afeat_host = t.copy()
            return
        Z, E, dev = t.shape[0], self.spec.embedding_dim, self.device
        self.atomic_features = torch.from_numpy(t).to(dev)
        self._afeat_host = t.copy()
        f = dict(dtype=torch.float32, device=dev)
        self._tab = {"emb": torch.empty(Z, E, **f), "d_emb": torch.empty(Z, E, **f), "G": torch.empty(Z + 3, D, **f)}
        for b in self._batches.values():
            for k in [k for k in b.graphs if k[-1] == TABLE_ROUTE]:
                del b.graphs[k]

    def _table_route(self) -> Optional[str]:
        """Route of a batch that arrives as atomic numbers: TABLE_ROUTE for a cgcnn model (which then needs the table)."""
        if self.spec.feature != "cgcnn":
            return None
        if self.atomic_features is None:
            raise ValueError("this feature='cgcnn' model got a batch of atomic numbers (CSR or device-gathered) before "
                             "its per-element feature table: call Engine.set_atomic_features(table) or pass "
                             "atomic_features= to the call that built the batches")
        return TABLE_ROUTE

    # ------------------------------------------------------------------ deterministic mode
    def _check_deterministic_support(self) -> None:
        """The deterministic mode exists for the default engine only: refuse every setting it cannot guarantee.  (Checked
        when training starts: inference is deterministic with every setting.)"""
        why = None
        if not (self.tc_dense and self.tc_la_fwd and self.tc_la_bwd):
            why = "the SIMT / round-1 kernels (SCANN_ENGINE=simt, SCANN_DENSE, SCANN_LA_FWD, SCANN_LA_BWD)"
        elif not self.use_chain or not self.use_chain2:
            why = "the unchained engine (SCANN_CHAIN=0 / SCANN_CHAIN2=0)"
        elif not self.use_wgrad_batch:
            why = "the per-layer weight-gradient kernels (SCANN_WGRAD_BATCH=0)"
        elif self.la_pipe != self.la_pipe_built:
            why = "the round-1 local-attention kernels (SCANN_LA_PIPE other than 15)"
        elif not self.noup_pipe:
            why = "the round-1 local-attention kernels (SCANN_NOUP_PIPE=0)"
        elif self.tile_stride_pref not in (0, 32):
            why = "tile slots other than 32 rows (SCANN_TILE_STRIDE)"
        elif self._skip:
            why = "SCANN_DEBUG_SKIP"
        if why is not None:
            raise NotImplementedError("deterministic mode is not available with " + why)

    def _check_deterministic_batch(self, b: "Batch") -> None:
        if b.stride != 32:
            raise NotImplementedError(
                f"deterministic mode needs the 32-row pipelined pair plan: this batch has up to {b.N} neighbours per "
                "atom (at most 32 are supported)")

    # ------------------------------------------------------------------ helpers
    def _ev(self, name: str, begin: bool) -> None:
        """CUDA-event bracket around one kernel launch (only when ``self.prof`` is a dict)."""
        if self.prof is None:
            return
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(torch.cuda.current_stream(self.device))
        if begin:
            self.prof.setdefault(name, []).append([ev, None])
        else:
            self.prof[name][-1][1] = ev

    def prof_summary(self) -> Dict[str, Tuple[int, float]]:
        """name -> (launches, mean milliseconds); call after a synchronize."""
        out = {}
        for k, evs in (self.prof or {}).items():
            ms = [a.elapsed_time(b) for a, b in evs if b is not None]
            if ms:
                out[k] = (len(ms), float(np.mean(ms)))
        return out

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _adrop(self, training: bool, layer: int):
        """(control block, site) of the attention-probability Dropout(0.05) of ``use_drop`` models
        (attention.py:115-116,191-192); (NULL, 0) outside training."""
        if training and self.spec.use_drop:
            return _p(self.adam_scalars, 12), 64 + layer
        return 0, 0

    def _pdl(self, on: bool) -> None:
        """Programmatic dependent launch for the following kernel launches of this thread.  Only switched
        on between two kernels of this library on the same stream (never right after a memset, a torch
        kernel or an event join)."""
        lib.scann_set_pdl(1 if (on and self.use_pdl) else 0)

    def w(self, name: str, off: int = 0) -> int:
        return _p(self.params, self.layout[name].offset + off)

    def wT(self, name: str, off: int = 0) -> int:
        return _p(self.paramsT, self.layout[name].offset + off)

    def gw(self, name: str, off: int = 0) -> int:
        return _p(self.grads, self.layout[name].offset + off)

    def check_status(self) -> None:
        if self.p2p is not None and float(self.p2p.sums[3].item()) != 0.0:
            self.p2p.sums[3] = 0.0
            raise _abi.ScannAbiError("peer-memory gradient exchange: a flag wait gave up (a peer rank is not taking part)")
        words = self.status.cpu().tolist()
        s = words[0]
        if s:
            self.status.zero_()
            msgs = [m for b, m in ERR_BITS.items() if s & b]
            if s & 16:
                msgs.append("wait site %d, CTA %d, tile %d, stage %d" % tuple(words[1:5]))
            raise _abi.ScannAbiError("device status: " + "; ".join(msgs))

    def set_params(self, arena: np.ndarray) -> None:
        self.params.copy_(torch.from_numpy(np.ascontiguousarray(arena, np.float32)))
        self._wimg_dirty = True

    def get_params(self) -> np.ndarray:
        return self.params.cpu().numpy()

    # ------------------------------------------------------------------ inputs
    def load_batch(self, inputs: Dict[str, object], plan: bool = True, pairs_hint: Optional[int] = None) -> Batch:
        """Stage one padded batch (reference layout, scann/utils/datagenerator.py:123-135) in the
        persistent device buffers of its shape class and build its pair plan.  Host arrays go through
        pinned staging buffers; CUDA tensors / ``__dlpack__`` objects are copied device-to-device.
        Buffers are persistent per (B, M, N, tile capacity) so that a captured CUDA graph can be
        replayed on every batch of that shape."""
        inputs = {k: import_tensor(v) for k, v in inputs.items()}     # DLPack capsules / exporters -> torch views
        nb = inputs["neighbors"]
        B, M, N = (int(s) for s in nb.shape)
        nmask_in = inputs["neighbor_mask"]
        P_host = int(np.count_nonzero(nmask_in)) if isinstance(nmask_in, np.ndarray) else None
        if P_host is None:
            P_host = pairs_hint
        b = self._get_batch(B, M, N, P_host)
        b.P_host = P_host
        b.h2d_bytes = 0
        b.route = None
        dev = self.device
        key = (B, M, N, b.tile_cap, b.tile_rows, b.stride)

        def put(dst: torch.Tensor, x, name):
            if isinstance(x, torch.Tensor):
                t = x
            else:
                a = np.ascontiguousarray(x)
                if a.dtype == np.bool_:
                    a = a.view(np.uint8)
                want = {torch.int32: np.int32, torch.uint8: np.uint8, torch.float32: np.float32}[dst.dtype]
                if a.dtype != want:
                    a = (a != 0).astype(np.uint8) if want is np.uint8 else a.astype(want)
                slot = self._pinned.get((name, key))
                if slot is None:
                    slot = self._pinned[(name, key)] = [torch.empty(dst.shape, dtype=dst.dtype).pin_memory(), None]
                pin, ev = slot
                if ev is not None:
                    ev.synchronize()            # the previous async copy out of this buffer has finished
                pin.numpy()[...] = a.reshape(pin.shape)
                dst.copy_(pin, non_blocking=True)
                slot[1] = torch.cuda.Event()
                slot[1].record(torch.cuda.current_stream(dev))
                b.h2d_bytes += a.nbytes
                return
            if t.numel() != dst.numel():
                raise ValueError(f"{name}: expected {dst.numel()} elements, got {t.numel()}")
            if dst.dtype == torch.uint8 and t.dtype not in (torch.uint8, torch.bool):
                t = t != 0
            dst.copy_(t.reshape(dst.shape), non_blocking=True)

        cg = self.spec.feature == "cgcnn"         # "atomic" then holds [B,M,92] feature vectors (datagenerator.py:109-110)
        items = [("atomic92" if cg else "atomic", inputs["atomic"]), ("atom_mask", inputs["atom_mask"]), ("nbr", nb),
                 ("nmask", nmask_in),
                 ("weight", inputs["neighbor_weight"]), ("dist", inputs["neighbor_distance"])]
        if self.spec.use_ring:
            items.append(("ring", inputs["ring_aromatic"]))
        if all(isinstance(x, np.ndarray) for _, x in items):
            # host arrays: fill the pinned mirror now, one asynchronous copy later (_flush_host)
            self._wait_pin(b)
            for name, x in items:
                dst = b.pin_np[name]
                a = x.view(np.uint8) if x.dtype == np.bool_ else x
                if dst.dtype == np.uint8 and a.dtype != np.uint8:
                    a = a != 0
                if a.size != dst.size:
                    raise ValueError(f"{name}: expected {dst.size} elements, got {a.size}")
                np.copyto(dst, a.reshape(dst.shape), casting="unsafe")
                b.h2d_bytes += x.nbytes
            b.host_dirty = True
        else:
            for name, x in items:
                put(getattr(b, name), x, name)
        if plan:
            self._plan(b)
        return b

    def _get_batch(self, B: int, M: int, N: int, P_host: Optional[int]) -> Batch:
        """Persistent device buffers of the shape class (B, M, N, tile capacity, tile layout)."""
        R = B * M
        P = P_host if P_host is not None else B * M * N
        ngroups = (R + PLAN_GSZ - 1) // PLAN_GSZ
        # rows per tile: fill whole waves of SMs (the kernels' cost per tile scales with its rows, and a
        # tile count just above a multiple of the SM count costs a whole extra round)
        tc = self.tc_la_fwd and self.tc_la_bwd
        pref = self.tile_stride_pref
        stride = 64 if (pref in (0, 64) and tc and N <= 32) else TILE
        # (32-row slots need the batched weight-gradient launch: the per-layer la_wgrad_tc kernels of the unbatched
        # variant only know 64 / 128-row slots)
        if N <= 32 and tc and self.use_chain and self.use_wgrad_batch and (
                pref == 32 or (pref == 0 and self.la_pipe and (self.spec.g_update or self.noup_pipe))):
            stride = 32
        tile_rows = stride
        # (the pipelined kernels on 32-row slots keep six tiles in flight per SM: full tiles, no wave balancing)
        if P_host is not None and self.balance_tiles and N <= 64 and stride != 32:
            slots = self.sm_count * (TILE // stride)
            waves = max(1, -(-P // (stride * slots)))      # more, smaller tiles only add per-tile latency (measured)
            tile_rows = min(stride, max(N, -(-P // (waves * slots)) + (N + 1) // 2))
            tile_rows = min(stride, (tile_rows + 7) // 8 * 8)          # quantised: few shape classes per data set
        # tile capacity: every non-final tile of a greedy group holds more than tile_rows-N rows
        # (and two consecutive tiles of a group together hold more than tile_rows rows)
        cap = (min(P // (tile_rows + 1 - N), 2 * P // tile_rows + 1) + ngroups + 1 if N <= 64
               else 2 * (P // TILE) + ngroups + 2)
        # shape classes are quantised (capacities on a geometric grid, ratio 1.25) so that a shuffled data set whose
        # batches differ a little in their pair counts maps onto a handful of persistent buffers / captured graphs
        tile_cap = 64
        while tile_cap < cap:
            tile_cap = (tile_cap * 5 // 4 + 63) // 64 * 64
        key = (B, M, N, tile_cap, tile_rows, stride)
        b = self._batches.get(key)
        if b is not None:
            self._batches.move_to_end(key)
        if b is None:
            while len(self._batches) >= self.max_shape_classes:      # least recently used class: buffers, graphs
                old_key, old = self._batches.popitem(last=False)
                self.shape_class_evictions += 1
                old.graphs.clear()
                for k in [k for k in self._pinned if k[1] == old_key]:
                    del self._pinned[k]
                live = {(x.R, x.B, x.rows) for x in self._batches.values()}
                for k in [k for k in self._ws if k[:3] not in live and k[:3] != (B * M, B, tile_cap * stride)]:
                    del self._ws[k]
            b = self._batches[key] = self._new_batch(B, M, N, tile_cap, ngroups, stride)
            b.tile_rows = tile_rows
            # rows of a tile slot that can hold pairs, rounded up to the MMA granularity: the N extent of the
            # local-attention MMAs (a wave-balanced plan fills ~40 of 64 rows)
            b.mma_rows = min(stride, (tile_rows + 15) // 16 * 16)
        return b

    def load_batch_csr(self, csr: Dict[str, object], target=None, plan: bool = True) -> Batch:
        """Stage one RAGGED batch (``DataIterator.csr_item`` of scann_b200/datagenerator.py): the CSR arrays travel
        in one host->device copy (valid atoms / pairs only) and ``scann_pack_batch`` expands them into the padded
        device buffers -- the device form of the reference's DataIterator.__getitem__."""
        route = self._table_route()
        sa, an = csr["struct_atom_off"], csr["atom_nbr_off"]
        B, M, N = len(sa) - 1, int(csr["M"]), int(csr["N"])
        idx = np.asarray(csr["nbr_idx"], np.int32)
        P_host = int(np.count_nonzero(idx != 1000))
        b = self._get_batch(B, M, N, P_host)
        b.P_host = P_host
        b.route = route
        segs = [("sa", np.asarray(sa, np.int32)), ("an", np.asarray(an, np.int32)), ("z", np.asarray(csr["z"], np.int32)),
                ("idx", idx), ("w", np.asarray(csr["nbr_w"], np.float32)), ("d", np.asarray(csr["nbr_d"], np.float32))]
        if self.spec.use_ring:
            segs.append(("ring", np.asarray(csr["ring"], np.int32).reshape(-1)))
        if target is not None:
            segs.append(("target", np.asarray(target, np.float32).reshape(-1)))
        offs, off = {}, 0
        for name, a in segs:
            offs[name] = off
            off += (a.nbytes + 15) // 16 * 16
        if getattr(b, "csr_pin", None) is None or b.csr_pin.numel() < off:
            cap = max(off, 4 * (B + 2 + 3 * b.R + 3 * b.R * N + b.R * 2 + B) + 256)
            b.csr_pin = torch.empty(cap, dtype=torch.uint8).pin_memory()
            b.csr_dev = torch.empty(cap, dtype=torch.uint8, device=self.device)
            b.csr_event = None
        if b.csr_event is not None:
            b.csr_event.synchronize()
        host = b.csr_pin.numpy()
        for name, a in segs:
            host[offs[name]:offs[name] + a.nbytes] = a.view(np.uint8).reshape(-1)
        main = torch.cuda.current_stream(self.device)
        if self.overlap_h2d:
            # the copy overlaps the previous step: it only has to wait for that step's scann_pack_batch
            cs = self.copy_stream
            if getattr(b, "csr_packed", None) is not None:
                cs.wait_event(b.csr_packed)
            with torch.cuda.stream(cs):
                b.csr_dev[:off].copy_(b.csr_pin[:off], non_blocking=True)
                b.csr_event = torch.cuda.Event()
                b.csr_event.record(cs)
            main.wait_event(b.csr_event)
        else:
            b.csr_dev[:off].copy_(b.csr_pin[:off], non_blocking=True)
            b.csr_event = torch.cuda.Event()
            b.csr_event.record(main)
        b.h2d_bytes = off
        self._pack_csr(b, b.csr_dev, offs)
        if self.overlap_h2d:
            b.csr_packed = torch.cuda.Event()
            b.csr_packed.record(main)
        if plan:
            self._plan(b)
        return b

    def load_batch_device_csr(self, csr: Dict[str, object], M: Optional[int] = None, N: Optional[int] = None,
                              plan: bool = True) -> Batch:
        """``load_batch_csr`` for a CSR batch that is already on the device (``voronoi.NeighborSelection.csr``): one
        blob ``csr["blob"]`` with the byte offsets ``csr["offsets"]`` (keys sa, an, z, idx, w, d) and the host sizes
        ``B`` / ``M`` / ``N`` / ``P``.  ``M`` / ``N`` may be raised above the batch's own (shape classes); the padding
        is masked.  Nothing crosses to or from the host."""
        route = self._table_route()
        B, P = int(csr["B"]), int(csr["P"])
        M = int(csr["M"]) if M is None else int(M)
        N = int(csr["N"]) if N is None else int(N)
        if M < int(csr["M"]) or N < int(csr["N"]):
            raise ValueError(f"M={M}, N={N} below the batch's own {csr['M']}, {csr['N']}")
        b = self._get_batch(B, M, N, P)
        b.P_host = P
        b.h2d_bytes = 0
        b.route = route
        self._pack_csr(b, csr["blob"], csr["offsets"])
        if plan:
            self._plan(b)
        return b

    def load_batch_gather(self, data, start: int, B: int, M: int, N: int, P: int, plan: bool = True) -> Batch:
        """Batch of structures ``data.perm[start:start + B]`` of a device-resident data set
        (``datagenerator.DeviceDataIterator``), padded by ``scann_gather_batch`` into the buffers of the shape class
        ``(B, M, N, P)`` -- the exact sizes of the batch, so that it shares the class and the captured graphs of the
        same structures loaded by ``load_batch_csr``.  The targets go to ``b.target``.  Nothing crosses to or from the
        host."""
        route = self._table_route()
        B, M, N, P = int(B), int(M), int(N), int(P)
        if B <= 0 or M <= 0 or N <= 0:
            raise ValueError(f"gather_batch: bad shape B={B} M={M} N={N}")
        if start < 0 or start + B > data.perm.numel():
            raise ValueError(f"gather_batch: structures {start}..{start + B} outside the permutation of "
                             f"{data.perm.numel()}")
        b = self._get_batch(B, M, N, P)
        b.P_host = P
        b.h2d_bytes = 0
        b.route = route
        b.host_dirty = False            # the pinned mirror is stale: it must not be copied over what is gathered here
        use_ring = self.spec.use_ring
        if use_ring and data.ring is None:
            raise ValueError("this model reads ring / aromatic flags: the data set has none (use_ring=False)")
        self._ev("gather_batch", True)
        check(lib.scann_gather_batch(_p(data.struct_atom_off), _p(data.atom_nbr_off), _p(data.z), _p(data.nbr_idx),
                                     _p(data.nbr_w), _p(data.nbr_d), _p(data.ring) if use_ring else 0, _p(data.target),
                                     _p(data.perm, start), B, M, N, _p(b.atomic), _p(b.atom_mask), _p(b.nbr),
                                     _p(b.nmask), _p(b.weight), _p(b.dist), _p(b.ring), _p(b.target), self._stream()),
              "gather_batch")
        self._ev("gather_batch", False)
        self.launches += 1
        if plan:
            self._plan(b)
        return b

    def _pack_csr(self, b: Batch, blob: torch.Tensor, offs: Dict[str, int]) -> None:
        """CSR blob on the device -> the padded buffers of the batch's shape class (scann_pack_batch)."""
        b.host_dirty = False            # the pinned mirror is stale: it must not be copied over what is packed here
        check(lib.scann_pack_batch(_p(blob), offs["sa"], offs["an"], offs["z"], offs["idx"], offs["w"], offs["d"],
                                   offs.get("ring", -1), offs.get("target", -1), b.B, b.M, b.N, _p(b.atomic),
                                   _p(b.atom_mask), _p(b.nbr), _p(b.nmask), _p(b.weight), _p(b.dist), _p(b.ring),
                                   _p(b.target), self._stream()), "pack_batch")
        self.launches += 1

    def _new_batch(self, B: int, M: int, N: int, tile_cap: int, ngroups: int, stride: int = TILE) -> Batch:
        dev = self.device
        b = Batch()
        b.B, b.M, b.N, b.R, b.tile_cap, b.ngroups = B, M, N, B * M, tile_cap, ngroups
        b.stride = stride
        rows = b.rows = tile_cap * stride
        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        # every host-provided array lives in ONE device blob mirrored by ONE pinned host blob: a step's inputs
        # (and its targets) travel in a single host->device copy instead of seven
        fields = [("atomic", torch.int32, b.R), ("atom_mask", torch.uint8, b.R), ("nbr", torch.int32, b.R * N),
                  ("nmask", torch.uint8, b.R * N), ("weight", torch.float32, b.R * N), ("dist", torch.float32, b.R * N),
                  ("target", torch.float32, B)]
        if self.spec.use_ring:
            fields.append(("ring", torch.float32, b.R * 2))
        if self.spec.feature == "cgcnn":
            fields.append(("atomic92", torch.float32, b.R * 92))
        off, offs = 0, {}
        for name, dt, n in fields:
            offs[name] = off
            off += (n * torch.empty((), dtype=dt).element_size() + 255) // 256 * 256
        b.blob = torch.zeros(off, dtype=torch.uint8, device=dev)
        b.blob_pin = torch.zeros(off, dtype=torch.uint8).pin_memory()
        b.pin_np, b.pin_event, b.host_dirty = {}, None, False
        b.ring = None
        for name, dt, n in fields:
            nb = n * torch.empty((), dtype=dt).element_size()
            setattr(b, name, b.blob[offs[name]:offs[name] + nb].view(dt))
            b.pin_np[name] = b.blob_pin[offs[name]:offs[name] + nb].view(dt).numpy()
        b.cnt = torch.empty(b.R, **i32)
        b.rowptr = torch.empty(b.R, **i32)
        b.tile_a0 = torch.empty(tile_cap, **i32)
        b.tile_a1 = torch.empty(tile_cap, **i32)
        b.ntiles = torch.zeros(1, **i32)
        b.pair_c = torch.empty(rows, **i32)
        b.pair_j = torch.empty(rows, **i32)
        b.pair_slot = torch.empty(rows, **i32)
        b.pair_d = torch.empty(rows, **f32)
        b.pair_w = torch.empty(rows, **f32)
        b.valid_rows = torch.empty(rows, **i32)
        b.valid_j = torch.empty(rows, **i32)
        b.nvalid = torch.zeros(1, **i32)
        # 4 ints per plan group (four-kernel form) + the 64-bit look-back words of the one-launch form, which rely
        # on the buffer being zero when it is first used (scann_plan_build)
        b.scratch = torch.zeros(6 * ngroups + 16, **i32)
        b.inv_ptr = None            # inverse neighbour CSR (deterministic mode, scann_plan_inverse)
        # local-attention scores (predict_step(local_attention=...)), allocated when first requested: [L, rows, 8] in
        # plan order as the kernels store them, and per layout the unpacked copy
        b.attn = None
        b.scores = {}
        b.graphs = {}
        return b

    def set_target(self, b: Batch, y_true) -> None:
        if isinstance(y_true, torch.Tensor):
            self._flush_host(b)         # the blob copy would overwrite the target region
            b.target.copy_(y_true.reshape(-1), non_blocking=True)
            return
        a = np.asarray(y_true, np.float32).reshape(-1)
        if a.size != b.B:
            raise ValueError("target must have one value per structure")
        if not b.host_dirty:
            self._wait_pin(b)
        b.pin_np["target"][...] = a
        b.h2d_bytes += a.nbytes
        if b.host_dirty:
            return                      # travels with the inputs in the single blob copy
        b.target.copy_(torch.from_numpy(b.pin_np["target"]), non_blocking=True)
        b.pin_event = torch.cuda.Event()
        b.pin_event.record(torch.cuda.current_stream(self.device))

    def _wait_pin(self, b: Batch) -> None:
        """The previous asynchronous copy out of the pinned mirror has finished (it may be overwritten)."""
        if b.pin_event is not None:
            b.pin_event.synchronize()
            b.pin_event = None

    def _flush_host(self, b: Batch) -> None:
        """One host->device copy of everything load_batch / set_target staged in the pinned mirror."""
        if not b.host_dirty:
            return
        main = torch.cuda.current_stream(self.device)
        if self.overlap_h2d and not torch.cuda.is_current_stream_capturing():
            # copy stream: pinned mirror -> staging blob (overlaps the previous step's kernels); main stream:
            # staging blob -> the blob the captured graph reads (a ~1 us device copy)
            if getattr(b, "blob_stage", None) is None:
                b.blob_stage = torch.empty_like(b.blob)
                b.stage_event = None
            cs = self.copy_stream
            if b.stage_event is not None:
                cs.wait_event(b.stage_event)        # the previous hand-over out of the staging blob has finished
            with torch.cuda.stream(cs):
                b.blob_stage.copy_(b.blob_pin, non_blocking=True)
                b.pin_event = torch.cuda.Event()
                b.pin_event.record(cs)
            main.wait_event(b.pin_event)
            b.blob.copy_(b.blob_stage, non_blocking=True)
            b.stage_event = torch.cuda.Event()
            b.stage_event.record(main)
        else:
            b.blob.copy_(b.blob_pin, non_blocking=True)
            b.pin_event = torch.cuda.Event()
            b.pin_event.record(main)
        b.host_dirty = False

    def _plan(self, b: Batch) -> None:
        self._flush_host(b)
        check(lib.scann_plan_build(_p(b.nmask), _p(b.nbr), _p(b.dist), _p(b.weight), b.B, b.M, b.N, b.tile_cap,
                                   b.tile_rows, b.stride, _p(b.cnt), _p(b.rowptr), _p(b.tile_a0), _p(b.tile_a1), _p(b.ntiles),
                                   _p(b.pair_c), _p(b.pair_j), _p(b.pair_slot), _p(b.pair_d), _p(b.pair_w),
                                   _p(b.valid_rows), _p(b.valid_j), _p(b.nvalid), _p(b.scratch), b.scratch.numel(), _p(self.status),
                                   self._stream()), "plan_build")
        # one launch (look-back over the plan groups), or count / group / scan / fill with SCANN_LA4 bit 5
        self.launches += 4 if (self.la_groups4 & 32) else 1
        if self.deterministic and b.stride == 32:
            if b.inv_ptr is None:
                i32 = dict(dtype=torch.int32, device=self.device)
                b.inv_ptr = torch.empty(b.R + 1, **i32)
                b.inv_idx = torch.empty(b.rows, **i32)
                b.inv_cnt = torch.empty(b.R, **i32)
                b.inv_tmp = torch.empty(b.rows, **i32)
            check(lib.scann_plan_inverse(_p(b.ntiles), b.stride, b.rows, _p(b.pair_c), _p(b.pair_j), b.R, _p(b.inv_ptr),
                                         _p(b.inv_idx), _p(b.inv_cnt), _p(b.inv_tmp), self._stream()), "plan_inverse")
            self.launches += 4

    # ------------------------------------------------------------------ workspaces
    def _workspace(self, b: Batch, training: bool) -> dict:
        key = (b.R, b.B, b.rows, training)          # workspaces depend on the capacity, not on tile_rows
        ws = self._ws.get(key)
        if ws is not None:
            return ws
        dev = self.device
        L = self.spec.n_attention
        R, rows = b.R, b.rows
        f = dict(dtype=torch.float32, device=dev)
        ws = {}
        nsave = L + 1 if training else 2
        ws["g"] = [torch.empty(rows, D, **f) for _ in range(nsave)] if self.spec.g_update else []
        if not self.spec.g_update and not training and self.noup_pipe and b.stride == 32:
            ws["gsave"] = [torch.empty(rows, D, **f)]         # g' of the current layer (pipelined attention kernel)
        ws["x"] = [torch.empty(R, D, **f) for _ in range(L + 1 if training else 2)]
        nl = L if training else 1
        ws["proj"] = [torch.empty(R, 3 * D, **f) for _ in range(nl)]
        ws["h"] = [torch.empty(R, D, **f) for _ in range(nl)]
        ws["h1"] = [torch.empty(R, D, **f) for _ in range(nl)]
        if training:
            ws["t0"] = torch.empty(R, D, **f)
            ws["ctxpre"] = [torch.empty(R, D, **f) for _ in range(L)]
            ws["t1"] = [torch.empty(R, D, **f) for _ in range(L)]
            ws["v2"] = [torch.empty(R, D, **f) for _ in range(L)]
            ws["ta"] = torch.empty(R, D, **f)
            if self.tc_la_bwd:
                if self.spec.g_update:
                    ws["pre"] = [torch.empty(rows, D, **f) for _ in range(L)]     # filter_geo pre-activation -> d_pre
                else:
                    ws["gsave"] = [torch.empty(rows, D, **f) for _ in range(L)]   # g' = swish(rbf Wf + bf) * w
                ws["kk"] = [torch.empty(rows, D, **f) for _ in range(L)]      # keys -> d_k
            ws["ctxg"] = torch.empty(b.B, D, **f)
            ws["tb"] = torch.empty(b.B, D, **f)
            # backward temporaries
            for k in ("dx", "d_h", "d_ctx", "d_ta"):
                ws[k] = torch.empty(R, D, **f)
            for k in ("d_v2", "d_v2m", "d_t1", "dq"):        # read by the weight-gradient kernels
                ws[k] = [torch.empty(R, D, **f) for _ in range(L)]
            ws["scat_all"] = torch.empty(L, 3, R, D, **f)    # s_pre, t_scatter, dx_scatter per layer, zeroed once
            ws["scat"] = [ws["scat_all"][l] for l in range(L)]
            ws["dg"] = [torch.empty(rows, D, **f) for _ in range(2)]
            ws["d_qk"] = torch.empty(R, 2 * D, **f)
            ws["d_tb"] = torch.empty(b.B, D, **f)
            ws["dy"] = torch.empty(b.B, **f)
            ws["wpart"] = torch.empty(self.la_grid, 2, D, D, **f)
            ws["G"] = torch.empty(self.spec.n_atoms + 3, D, **f)
        if training and self.deterministic:
            self._det_workspace(b, ws)
        ws["xa"] = torch.empty(R, D, **f)
        ws["qk"] = torch.empty(R, 2 * D, **f)
        ws["ga"] = torch.empty(R, **f)
        ws["y"] = torch.empty(b.B, **f)
        self._ws[key] = ws
        return ws

    def _det_workspace(self, b: Batch, ws: dict) -> None:
        """Per-pair buffer and per-CTA slot arrays of the deterministic mode, and the table of slot arrays that
        scann_slot_reduce adds into the gradient arena before the optimiser."""
        sp, dev = self.spec, self.device
        L, R, G = sp.n_attention, b.R, self.la_grid
        f = dict(dtype=torch.float32, device=dev)
        ws["pairbuf"] = torch.empty(b.rows, D, **f)                   # d_a * g' per pair, reused by every layer
        ws["dbk_slots"] = torch.empty(L, G, D, **f)
        if sp.g_update:
            ws["lng_slots"] = torch.empty(L, G, 2 * D, **f)           # layer_norm_g gamma | beta
        # CTAs of the chained launches over R rows: the warp-specialised form up to one wave, else the round-1 form
        cg = (lib.scann_dense_chain2_grid(R) if self.use_chain2 and R <= self.chain2_max_rows
              else lib.scann_dense_chain_grid(R))
        ws["ln_slots"] = torch.empty(L, 2, 2, cg, D, **f)             # [layer][layer_norm, residual_norm][gamma, beta]
        ws["wg_slots"] = torch.empty(G, 2, D * D, **f)
        ws["wg_bslots"] = torch.empty(G, 2, D, **f)
        gi = G * self.gi_bwd_mult
        gslot = 2 * N_RBF * D + 2 * D                                  # geometry initialisation: dWd | dWw | dbd | dbw
        nslot = (N_RBF + 1) * D                                        # g_update=False filter: dWf | dbf
        if sp.g_update:
            ws["gi_slots"] = torch.empty(2 * gi, gslot, **f)
        else:
            ws["noup_slots"] = torch.empty(L, 2 * gi, nslot, **f)
        kin = sp.embedding_dim + (10 if sp.use_ring else 0)
        if sp.feature == "cgcnn":
            ws["cg_slots"] = torch.empty((R + 31) // 32, (kin + 1) * D, **f)    # dense_embed kernel rows | bias
        else:
            ns = lib.scann_embed_backward_det_slots(R)
            ws["emb_slots"] = torch.empty(ns, sp.n_atoms + 3, D, **f)
        ws["head_slots"] = torch.empty(b.B, D, **f)                   # predict_property kernel, per structure
        ws["head_bslots"] = torch.empty(b.B, **f)                     # predict_property bias, per structure
        ws["reg_slots"] = torch.empty(1184, **f)
        ents = []

        def add(slots: torch.Tensor, nslots: int, count: int, ld: int, dst: int, off: int = 0) -> None:
            e = _abi.SlotSum()
            e.slots, e.dst, e.nslots, e.count, e.ld, e.pad = _p(slots, off), dst, nslots, count, ld, 0
            ents.append(e)

        for l in range(L):
            la = layer_name("local_attention", l)
            rn = layer_name("residual_norm", l)
            add(ws["dbk_slots"][l], G, D, D, self.gw(f"{la}/key/bias"))
            if sp.g_update:
                add(ws["lng_slots"][l], G, D, 2 * D, self.gw(f"{la}/layer_norm_g/gamma"))
                add(ws["lng_slots"][l], G, D, 2 * D, self.gw(f"{la}/layer_norm_g/beta"), D)
            else:
                add(ws["noup_slots"][l], 2 * gi, N_RBF * D, nslot, self.gw(f"{la}/filter_geo/kernel"))
                add(ws["noup_slots"][l], 2 * gi, D, nslot, self.gw(f"{la}/filter_geo/bias"), N_RBF * D)
            add(ws["ln_slots"][l, 0, 0], cg, D, D, self.gw(f"{la}/layer_norm/gamma"))
            add(ws["ln_slots"][l, 0, 1], cg, D, D, self.gw(f"{la}/layer_norm/beta"))
            if sp.use_attn_norm:
                add(ws["ln_slots"][l, 1, 0], cg, D, D, self.gw(f"{rn}/layer_norm/gamma"))
                add(ws["ln_slots"][l, 1, 1], cg, D, D, self.gw(f"{rn}/layer_norm/beta"))
        if sp.g_update:
            gs = ws["gi_slots"]
            add(gs, 2 * gi, N_RBF * D, gslot, self.gw("neighbor_d/kernel"))
            add(gs, 2 * gi, N_RBF * D, gslot, self.gw("neighbor_w/kernel"), N_RBF * D)
            add(gs, 2 * gi, D, gslot, self.gw("neighbor_d/bias"), 2 * N_RBF * D)
            add(gs, 2 * gi, D, gslot, self.gw("neighbor_w/bias"), 2 * N_RBF * D + D)
        i_cg = len(ents)
        if sp.feature == "cgcnn":
            cs = ws["cg_slots"]
            add(cs, cs.shape[0], kin * D, (kin + 1) * D, self.gw("dense_embed/kernel"))
            add(cs, cs.shape[0], D, (kin + 1) * D, self.gw("dense_embed/bias"), kin * D)
        add(ws["head_slots"], b.B, D, D, self.gw("predict_property/kernel"))
        add(ws["head_bslots"], b.B, 1, 1, self.gw("predict_property/bias"))

        def table(es):
            arr = (_abi.SlotSum * len(es))(*es)
            return torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(dev), len(es)
        ws["slot_table"], ws["slot_count"] = table(ents)
        ws["slot_max"] = max(e.count for e in ents)
        if sp.feature == "cgcnn":
            # table route: dense_embed's gradients come out of the embedding backward itself, cg_slots are not written
            ws["slot_table_" + TABLE_ROUTE], ws["slot_count_" + TABLE_ROUTE] = table(ents[:i_cg] + ents[i_cg + 2:])

    def _ln_grads(self, ws: dict, l: int, which: int, name: str) -> dict:
        """dgamma / dbeta of a LayerNorm-backward chain step: the gradient arena, or the slot arrays of the deterministic
        mode (which: 0 the attention output's LayerNorm, 1 the ResidualNorm's)."""
        if self.deterministic:
            return dict(dgamma=_p(ws["ln_slots"][l, which, 0]), dbeta=_p(ws["ln_slots"][l, which, 1]))
        return dict(dgamma=self.gw(f"{name}/layer_norm/gamma"), dbeta=self.gw(f"{name}/layer_norm/beta"))

    # ------------------------------------------------------------------ thin kernel wrappers
    def _dense(self, A, lda, W, bias, kblk, nblk, R, C, ldc, mode=0, resid=None, ldres=D, pre_in=None, pre_out=None,
               gamma=0, beta=0):
        fn = lib.scann_dense_forward_tc if self.tc_dense else lib.scann_dense_forward
        check(fn(ptr_array(A), lda, ptr_array(W), ptr_array(bias) if bias else None, kblk, nblk,
                                      R, C, ldc, mode, _p(resid), ldres, _p(pre_in), _p(pre_out), gamma, beta,
                                      self._stream()), "dense_forward")
        self.launches += 1

    def _weight_images(self, stream: Optional[int] = None) -> None:
        """Operand images of every 128x128 weight block (scann_weight_images) from the current parameters."""
        if not self.use_chain2:
            return
        check(lib.scann_weight_images(_p(self.params), _p(self.tblocks), self.tblocks.numel(), self._wimg_base,
                                      self._stream() if stream is None else stream), "weight_images")
        self.launches += 1
        self._wimg_dirty = False

    def _wimg_ptr(self, p: int) -> int:
        """Weight image of the block a ``w()`` pointer (orientation 0: x @ W) or a ``wT()`` pointer (orientation 1:
        x @ W^T) addresses."""
        nbytes = 4 * self.layout.total
        for base, orient in ((self.params.data_ptr(), 0), (self.paramsT.data_ptr(), 1)):
            if base <= p < base + nbytes:
                return self._wimg_base + (self._wimg_index[(p - base) // 4] * 2 + orient) * 131072
        raise KeyError("not a weight block of the parameter arena")

    def _chain(self, steps, R):
        """One scann_dense_chain launch: ``steps`` is a list of ChainStep (see include/scann_b200.h).  Up to 64 rows
        per SM the warp-specialised form runs (scann_dense_chain2: weight pointers replaced by their operand images)."""
        if "chain" in self._skip:
            return
        if self.use_chain2 and R <= self.chain2_max_rows:
            for s in steps:
                for kb in range(s.kblk):
                    s.W[kb] = self._wimg_ptr(s.W[kb])
            arr = (ChainStep * len(steps))(*steps)
            fn = lib.scann_dense_chain2_det if self.deterministic else lib.scann_dense_chain2
            check(fn(ctypes.cast(arr, ctypes.c_void_p), len(steps), R, _p(self.status), self._stream()), "dense_chain2")
            self.launches += 1
            return
        arr = (ChainStep * len(steps))(*steps)
        fn = lib.scann_dense_chain_det if self.deterministic else lib.scann_dense_chain
        check(fn(ctypes.cast(arr, ctypes.c_void_p), len(steps), R, self._stream()), "dense_chain")
        self.launches += 1

    def _wgrad(self, A, lda, G, ldg, kblk, nblk, R, dW, db):
        check(lib.scann_dense_wgrad(ptr_array(A), lda, ptr_array(G), ldg, kblk, nblk, R, ptr_array(dW),
                                    ptr_array(db) if db else None, self._stream()), "dense_wgrad")
        self.launches += 1

    # ------------------------------------------------------------------ forward
    def _embed_forward(self, b: Batch, ws: dict, training: bool, st: int) -> None:
        """Input embedding + dense_embed (+ ring features, Dropout 0.1) -> x_0  (scann_model.py:361-374)."""
        sp = self.spec
        R, E = b.R, sp.embedding_dim
        ring = sp.use_ring
        cg = sp.feature == "cgcnn"
        if b.route == TABLE_ROUTE:
            # embed_atom over the per-element table once (emb_table = table @ W + b), then the lookup of row Z: the
            # arithmetic of each row is that of the padded route's per-atom rows, bit for bit
            Z, emb = self.atomic_features.shape[0], self._tab["emb"]
            check(lib.scann_cgcnn_embed_forward(_p(self.atomic_features), self.w("embed_atom/kernel"),
                                                self.w("embed_atom/bias"), Z, 92, E, _p(emb), st), "cgcnn_embed_forward")
            self.launches += 1
            check(lib.scann_embed_forward(_p(b.atomic), _p(b.ring) if ring else 0, R, E, Z, _p(emb),
                                          self.w("extra_embed/kernel") if ring else 0, self.w("extra_embed/bias") if ring else 0,
                                          self.w("dense_embed/kernel"), self.w("dense_embed/bias"),
                                          _p(ws["t0"]) if training else 0, _p(ws["x"][0]), _p(self.status),
                                          _p(self.adam_scalars, 8) if training else 0, 0, st), "embed_forward")
            self.launches += 1
            return
        if cg:
            if "emb_rows" not in ws:
                ws["emb_rows"] = torch.empty(R, E, dtype=torch.float32, device=self.device)
                ws["d_cat"] = torch.empty(R, 144, dtype=torch.float32, device=self.device)
            check(lib.scann_cgcnn_embed_forward(_p(b.atomic92), self.w("embed_atom/kernel"), self.w("embed_atom/bias"),
                                                R, 92, E, _p(ws["emb_rows"]), st), "cgcnn_embed_forward")
            self.launches += 1
        check(lib.scann_embed_forward(_p(b.atomic), _p(b.ring) if ring else 0, R, E, sp.n_atoms,
                                      0 if cg else self.w("embed_atom/embeddings"), self.w("extra_embed/kernel") if ring else 0,
                                      self.w("extra_embed/bias") if ring else 0,
                                      self.w("dense_embed/kernel"), self.w("dense_embed/bias"),
                                      _p(ws["t0"]) if training else 0, _p(ws["x"][0]), _p(self.status),
                                      _p(self.adam_scalars, 8) if training else 0, _p(ws["emb_rows"]) if cg else 0, st),
              "embed_forward")
        self.launches += 1

    def forward(self, b: Batch, training: bool = False, attn: Optional[torch.Tensor] = None, replan: bool = False,
                side_work=None):
        """Runs the whole graph; returns (y[B], ga[B*M]) device tensors (views of the workspace).  ``attn``
        ([L, rows, 8] fp32, or None): the local-attention kernels store every layer's softmax there, in pair-plan order.

        Two branches meet in front of the first per-atom projection: the pair plan (``replan``) and the geometry
        initialisation need the neighbour lists only, the weight operand images and the embedding need the atoms
        only.  With a side stream the second branch (and ``side_work()``: whatever else the caller wants enqueued
        there, e.g. the preparation of the backward pass) runs beside the first."""
        sp, st = self.spec, self._stream()
        self._flush_host(b)
        ws = self._workspace(b, training)
        L, R = sp.n_attention, b.R
        xs, gs = ws["x"], ws["g"]
        if training and not sp.g_update and not (self.use_chain and self.tc_la_bwd and self.use_wgrad_batch):
            raise NotImplementedError("training of g_update=False models needs the tensor-core engine "
                                      "(SCANN_ENGINE=tc, SCANN_CHAIN=1)")
        self._pdl(False)
        main = torch.cuda.current_stream(self.device)
        fork = self.use_side_stream and (replan or side_work is not None)
        embed_ev = None
        if fork:
            ev = torch.cuda.Event()
            ev.record(main)
            self.side_stream.wait_event(ev)
            with torch.cuda.stream(self.side_stream):
                sst = self.side_stream.cuda_stream
                if self._wimg_dirty or training:
                    self._weight_images(sst)
                self._embed_forward(b, ws, training, sst)
                embed_ev = torch.cuda.Event()
                embed_ev.record(self.side_stream)
                if side_work is not None:
                    side_work()
            if replan:
                self._plan(b)
        else:
            if replan:
                self._plan(b)
            if self._wimg_dirty or training:
                self._weight_images()
            self._embed_forward(b, ws, training, st)
            if side_work is not None:
                side_work()
        if sp.g_update and "geom_init" not in self._skip:
            check(lib.scann_geom_init_forward(_p(b.ntiles), self.la_grid * self.gi_fwd_mult, b.stride, _p(b.pair_c), _p(b.pair_d), _p(b.pair_w),
                                              _p(self.centers_d), _p(self.centers_w), self.w("neighbor_d/kernel"),
                                              self.w("neighbor_d/bias"), self.w("neighbor_w/kernel"),
                                              self.w("neighbor_w/bias"), _p(gs[0]), st), "geom_init_forward")
            self.launches += 1
        if embed_ev is not None:
            main.wait_event(embed_ev)         # x_0 and the weight images are ready
        if self.use_chain and (not training or self.tc_la_bwd):
            return self._forward_chained(b, ws, training, attn)    # (first launch without PDL, then switched on)
        self._pdl(not fork)
        for l in range(L):
            la = layer_name("local_attention", l)
            rn = layer_name("residual_norm", l)
            li = l if training else 0
            x_in = xs[l] if training else xs[l % 2]
            x_out = xs[l + 1] if training else xs[(l + 1) % 2]
            proj, h, h1 = ws["proj"][li], ws["h"][li], ws["h1"][li]
            fg = f"{la}/filter_geo/kernel"
            ctxpre = ws["ctxpre"][l] if training else None
            out = h if sp.use_attn_norm else x_out
            attn_l = _p(attn, l * b.rows * 8)
            if not sp.g_update:
                # SCANN without geometry update (attention.py:155): only the query block of proj is needed
                self._dense([_p(x_in)], D, [self.w(f"{la}/query/kernel")], [self.w(f"{la}/query/bias")], 1, 1, R,
                            _p(proj, 2 * D), 3 * D)
                check(lib.scann_la_nopair_forward(_p(b.cnt), _p(proj), R, self.w(f"{la}/layer_norm/gamma"),
                                                  self.w(f"{la}/layer_norm/beta"), 0, _p(out), st), "la_nopair")
                check(lib.scann_la_forward_noupdate_tc(
                    self.la_grid, b.stride, b.mma_rows, _p(b.ntiles), _p(b.tile_a0), _p(b.tile_a1), _p(b.cnt), _p(b.rowptr), _p(b.pair_c),
                    _p(b.pair_j), _p(x_in), _p(proj), _p(b.pair_d), _p(b.pair_w), _p(self.centers_d), self.w(fg),
                    self.w(f"{la}/filter_geo/bias"), self.w(f"{la}/key/kernel"), self.w(f"{la}/key/bias"),
                    self.w(f"{la}/layer_norm/gamma"), self.w(f"{la}/layer_norm/beta"), 0, _p(out), attn_l, 0, 0, *self._adrop(training, l), st),
                    "la_forward_noupdate_tc")
                self.launches += 2
                if sp.use_attn_norm:
                    self._dense([_p(h)], D, [self.w(f"{rn}/dense/kernel")], [self.w(f"{rn}/dense/bias")], 1, 1, R,
                                _p(h1), D, mode=1)
                    self._dense([_p(h1)], D, [self.w(f"{rn}/dense_1/kernel")], [self.w(f"{rn}/dense_1/bias")], 1, 1, R,
                                _p(x_out), D, mode=3, resid=h, gamma=self.w(f"{rn}/layer_norm/gamma"),
                                beta=self.w(f"{rn}/layer_norm/beta"))
                continue
            g_in = gs[l] if training else gs[l % 2]
            g_out = gs[l + 1] if training else gs[(l + 1) % 2]
            # per-atom projections [x@W1+bf | x@W3 | x@Wq+bq]
            self._dense([_p(x_in)], D, [self.w(fg, 0), self.w(fg, 2 * D * D), self.w(f"{la}/query/kernel")],
                        [self.w(f"{la}/filter_geo/bias"), 0, self.w(f"{la}/query/bias")], 1, 3, R, _p(proj), 3 * D)
            check(lib.scann_la_nopair_forward(_p(b.cnt), _p(proj), R, self.w(f"{la}/layer_norm/gamma"),
                                              self.w(f"{la}/layer_norm/beta"), _p(ctxpre), _p(out), st), "la_nopair")
            self._ev("la_forward", True)
            la_args = (_p(b.ntiles), _p(b.tile_a0), _p(b.tile_a1), _p(b.cnt),
                       _p(b.rowptr), _p(b.pair_c), _p(b.pair_j), _p(x_in), _p(proj), _p(g_in),
                       self.w(fg, D * D), self.w(f"{la}/key/kernel"), self.w(f"{la}/key/bias"),
                       self.w(f"{la}/layer_norm_g/gamma"), self.w(f"{la}/layer_norm_g/beta"),
                       self.w(f"{la}/layer_norm/gamma"), self.w(f"{la}/layer_norm/beta"),
                       _p(g_out), _p(ctxpre), _p(out), attn_l)
            if "la_fwd" in self._skip:
                pass
            elif self.tc_la_fwd:
                save = training and self.tc_la_bwd
                self._la_forward_tc(b, la_args, _p(ws["pre"][l]) if save else 0, _p(ws["kk"][l]) if save else 0,
                                    self._adrop(training, l), st)
                self.launches += 1
            else:
                check(lib.scann_la_forward(self.la_grid, *la_args, st), "la_forward")
            self._ev("la_forward", False)
            self.launches += 2
            if sp.use_attn_norm and "rn" not in self._skip:
                # ResidualNorm: LN(h + Dense(swish(Dense(h))))  (attention.py:25-40)
                self._dense([_p(h)], D, [self.w(f"{rn}/dense/kernel")], [self.w(f"{rn}/dense/bias")], 1, 1, R, _p(h1),
                            D, mode=1, pre_out=ws["t1"][l] if training else None)
                self._dense([_p(h1)], D, [self.w(f"{rn}/dense_1/kernel")], [self.w(f"{rn}/dense_1/bias")], 1, 1, R,
                            _p(x_out), D, mode=3, resid=h, pre_out=ws["v2"][l] if training else None,
                            gamma=self.w(f"{rn}/layer_norm/gamma"), beta=self.w(f"{rn}/layer_norm/beta"))
        x_last = xs[L] if training else xs[L % 2]
        self._dense([_p(x_last)], D, [self.w("after_Lc/kernel")], [self.w("after_Lc/bias")], 1, 1, R, _p(ws["xa"]), D,
                    mode=1, pre_out=ws["ta"] if training else None)
        self._dense([_p(ws["xa"])], D, [self.w("global_attention/query/kernel"), self.w("global_attention/key/kernel")],
                    [self.w("global_attention/query/bias"), self.w("global_attention/key/bias")], 1, 2, R,
                    _p(ws["qk"]), 2 * D)
        self._ev("ga_forward", True)
        check(lib.scann_ga_head_forward(_p(ws["qk"]), _p(b.atom_mask), b.B, b.M, int(sp.use_ga_norm),
                                        self.w("bf_property/kernel"), self.w("bf_property/bias"),
                                        self.w("predict_property/kernel"), self.w("predict_property/bias"),
                                        int(sp.mrelu_head), _p(ws["ga"]), _p(ws["y"]),
                                        _p(ws["ctxg"]) if training else 0, _p(ws["tb"]) if training else 0, st),
              "ga_head_forward")
        self._ev("ga_forward", False)
        self._pdl(False)
        self.launches += 1
        return ws["y"], ws["ga"]

    def _la_forward_tc(self, b: Batch, la_args, pre_out: int, k_out: int, adrop, st: int) -> None:
        """LocalAttention forward (g_update=True) of one layer: the pipelined kernels on 32-row plans (``la_pipe`` bits
        0 / 1), else the round-1 tensor-core kernels.  A half that is switched off is run by the round-1 kernels
        (development: both kernels of the old form run first, the selected pipelined half then rewrites its outputs)."""
        which = self.la_pipe & 3 if b.stride == 32 else 0
        if which != 3:
            check(lib.scann_la_forward_tc(self.la_grid, b.stride, b.mma_rows, *la_args, pre_out, k_out, *adrop, st),
                  "la_forward_tc")
        if which:
            (ntiles, _a0, _a1, _cnt, _rowptr, pair_c, pair_j, x_in, proj, g_in, W2, Wk, bk, gg, bg, gam, bet, g_out,
             ctxpre, out, attn) = la_args
            check(lib.scann_la_forward_pipe(self.la_grid, b.rows, which, ntiles, pair_c, pair_j, x_in, proj, g_in, W2, Wk, bk,
                                            gg, bg, gam, bet, g_out, ctxpre, out, attn, pre_out, k_out, *adrop,
                                            _p(self.status), st), "la_forward_pipe")

    def _forward_chained(self, b: Batch, ws: dict, training: bool, attn: Optional[torch.Tensor]):
        """Layers of the forward pass with the per-atom Dense layers fused (scann_dense_chain):
        [projections of layer 0] -> LA_0 -> [ResidualNorm_0 + projections of layer 1] -> LA_1 -> ... ->
        [ResidualNorm_{L-1} + after_Lc + GlobalAttention q/k] -> GA + head."""
        sp, st = self.spec, self._stream()
        L, R = sp.n_attention, b.R
        xs, gs = ws["x"], ws["g"]

        def bufs(l):
            li = l if training else 0
            x_in = xs[l] if training else xs[l % 2]
            x_out = xs[l + 1] if training else xs[(l + 1) % 2]
            h = ws["h"][li]
            return li, x_in, x_out, ws["proj"][li], h, ws["h1"][li], (h if sp.use_attn_norm else x_out)

        def proj_steps(l, src):
            """x @ [W1 | W3 | Wq] (+ biases) of layer l into its proj buffer; rows without a valid neighbour get
            context = q and out = LN(q).  ``src``: global tensor holding x_l, or None = resident image."""
            la = layer_name("local_attention", l)
            fg = f"{la}/filter_geo/kernel"
            li, _, _, proj, _, _, out = bufs(l)
            ctxpre = ws["ctxpre"][l] if training else None
            A = [_p(src)] if src is not None else []
            steps = []
            if sp.g_update:
                steps.append(chain_step(A=A, W=[self.w(fg, 0)], bias=self.w(f"{la}/filter_geo/bias"), C_=_p(proj), ldc=3 * D))
                steps.append(chain_step(W=[self.w(fg, 2 * D * D)], C_=_p(proj, D), ldc=3 * D))
                A = []
            steps.append(chain_step(A=A, W=[self.w(f"{la}/query/kernel")], bias=self.w(f"{la}/query/bias"),
                                    C_=_p(proj, 2 * D), ldc=3 * D, cnt=_p(b.cnt), np_ctx=_p(ctxpre), np_out=_p(out),
                                    gamma=self.w(f"{la}/layer_norm/gamma"), beta=self.w(f"{la}/layer_norm/beta")))
            return steps

        self._chain(proj_steps(0, xs[0]), R)
        self._pdl(True)
        for l in range(L):
            la = layer_name("local_attention", l)
            rn = layer_name("residual_norm", l)
            fg = f"{la}/filter_geo/kernel"
            li, x_in, x_out, proj, h, h1, out = bufs(l)
            ctxpre = ws["ctxpre"][l] if training else None
            attn_l = _p(attn, l * b.rows * 8)
            self._ev("la_forward", True)
            if "la_fwd" in self._skip:
                pass
            elif sp.g_update:
                g_in = gs[l] if training else gs[l % 2]
                g_out = gs[l + 1] if training else gs[(l + 1) % 2]
                save = training and self.tc_la_bwd
                self._la_forward_tc(b, (
                    _p(b.ntiles), _p(b.tile_a0), _p(b.tile_a1), _p(b.cnt), _p(b.rowptr),
                    _p(b.pair_c), _p(b.pair_j), _p(x_in), _p(proj), _p(g_in), self.w(fg, D * D),
                    self.w(f"{la}/key/kernel"), self.w(f"{la}/key/bias"), self.w(f"{la}/layer_norm_g/gamma"),
                    self.w(f"{la}/layer_norm_g/beta"), self.w(f"{la}/layer_norm/gamma"),
                    self.w(f"{la}/layer_norm/beta"), _p(g_out), _p(ctxpre), _p(out), attn_l),
                    _p(ws["pre"][l]) if save else 0, _p(ws["kk"][l]) if save else 0, self._adrop(training, l), st)
                self.launches += 2
            elif self.noup_pipe and b.stride == 32 and "gsave" in ws:
                # g_update = False on the pipelined attention kernel: g' written out, then read by TMA
                gbuf = ws["gsave"][l if training else 0]
                check(lib.scann_noupdate_geom_forward(
                    _p(b.ntiles), self.la_grid * self.gi_fwd_mult, b.stride, _p(b.pair_c), _p(b.pair_d), _p(b.pair_w),
                    _p(self.centers_d), self.w(fg), self.w(f"{la}/filter_geo/bias"), _p(gbuf), st), "noupdate_geom_forward")
                check(lib.scann_la_forward_pipe(
                    self.la_grid, b.rows, 2, _p(b.ntiles), _p(b.pair_c), _p(b.pair_j), _p(x_in), _p(proj), 0, 0,
                    self.w(f"{la}/key/kernel"), self.w(f"{la}/key/bias"), 0, 0, self.w(f"{la}/layer_norm/gamma"),
                    self.w(f"{la}/layer_norm/beta"), _p(gbuf), _p(ctxpre), _p(out), attn_l, 0,
                    _p(ws["kk"][l]) if training else 0, *self._adrop(training, l), _p(self.status), st),
                    "la_forward_pipe")
                self.launches += 2
            else:
                check(lib.scann_la_forward_noupdate_tc(
                    self.la_grid, b.stride, b.mma_rows, _p(b.ntiles), _p(b.tile_a0), _p(b.tile_a1), _p(b.cnt), _p(b.rowptr),
                    _p(b.pair_c), _p(b.pair_j), _p(x_in), _p(proj), _p(b.pair_d), _p(b.pair_w), _p(self.centers_d),
                    self.w(fg), self.w(f"{la}/filter_geo/bias"), self.w(f"{la}/key/kernel"), self.w(f"{la}/key/bias"),
                    self.w(f"{la}/layer_norm/gamma"), self.w(f"{la}/layer_norm/beta"), _p(ctxpre), _p(out), attn_l,
                    _p(ws["gsave"][l]) if training else 0, _p(ws["kk"][l]) if training else 0, *self._adrop(training, l), st),
                    "la_forward_noupdate_tc")
                self.launches += 1
            self._ev("la_forward", False)
            steps = []
            src = x_out                       # where x_{l+1} lives if no step of this chain produces it
            if sp.use_attn_norm and "rn" not in self._skip:
                # ResidualNorm: LN(h + Dense(swish(Dense(h))))  (attention.py:25-40)
                steps.append(chain_step(A=[_p(h)], W=[self.w(f"{rn}/dense/kernel")], bias=self.w(f"{rn}/dense/bias"),
                                        mode=1, pre_out=_p(ws["t1"][l]) if training else 0, C_=_p(h1), to_image=True))
                steps.append(chain_step(W=[self.w(f"{rn}/dense_1/kernel")], bias=self.w(f"{rn}/dense_1/bias"),
                                        resid=_p(h), mode=3, pre_out=_p(ws["v2"][l]) if training else 0,
                                        gamma=self.w(f"{rn}/layer_norm/gamma"), beta=self.w(f"{rn}/layer_norm/beta"),
                                        C_=_p(x_out), to_image=True,
                                        drop=_p(self.adam_scalars, 8) if training else 0, drop_site=1 + l))
                src = None
            if l + 1 < L:
                steps += proj_steps(l + 1, src)
            else:
                A = [_p(src)] if src is not None else []
                steps.append(chain_step(A=A, W=[self.w("after_Lc/kernel")], bias=self.w("after_Lc/bias"), mode=1,
                                        pre_out=_p(ws["ta"]) if training else 0, C_=_p(ws["xa"]), to_image=True))
                steps.append(chain_step(W=[self.w("global_attention/query/kernel")],
                                        bias=self.w("global_attention/query/bias"), C_=_p(ws["qk"]), ldc=2 * D))
                steps.append(chain_step(W=[self.w("global_attention/key/kernel")],
                                        bias=self.w("global_attention/key/bias"), C_=_p(ws["qk"], D), ldc=2 * D))
            self._chain(steps, R)
        self._ev("ga_forward", True)
        check(lib.scann_ga_head_forward(_p(ws["qk"]), _p(b.atom_mask), b.B, b.M, int(sp.use_ga_norm),
                                        self.w("bf_property/kernel"), self.w("bf_property/bias"),
                                        self.w("predict_property/kernel"), self.w("predict_property/bias"),
                                        int(sp.mrelu_head), _p(ws["ga"]), _p(ws["y"]),
                                        _p(ws["ctxg"]) if training else 0, _p(ws["tb"]) if training else 0, st),
              "ga_head_forward")
        self._ev("ga_forward", False)
        self._pdl(False)
        self.launches += 1
        return ws["y"], ws["ga"]

    # ------------------------------------------------------------------ backward
    def backward(self, b: Batch, target: torch.Tensor) -> None:
        """Accumulates G = sum_b (y_b - t_b) dy_b/dtheta into the (pre-zeroed) gradient arena and
        the SSE into its tail.  ``forward(b, training=True)`` must have run on the same batch.

        The chain of input gradients (dense_tc / LayerNorm backward / local-attention backward) is the
        critical path and runs on the current stream; every weight-gradient kernel only feeds the
        optimiser, so they are issued on a side stream (fork / join through events, captured into the
        same CUDA graph) and overlap the next layer's chain.  Buffers read by the side stream are
        per layer."""
        sp, st = self.spec, self._stream()
        ws = self._workspace(b, True)
        L, R, n = sp.n_attention, b.R, self.layout.total
        main = torch.cuda.current_stream(self.device)
        side = self.side_stream if self.use_side_stream else main
        sst = side.cuda_stream

        def fork():                      # side stream may start once everything issued so far is done
            if side is not main:
                ev = torch.cuda.Event()
                ev.record(main)
                side.wait_event(ev)

        def wgrad(A, lda, G, ldg, kblk, nblk, rows, dW, db):
            check(lib.scann_dense_wgrad(ptr_array(A), lda, ptr_array(G), ldg, kblk, nblk, rows, ptr_array(dW),
                                        ptr_array(db) if db else None, sst), "dense_wgrad")
            self.launches += 1

        if side is not main and self._prep_event is not None:
            main.wait_event(self._prep_event)        # transposed weights + zeroed scatter buffers are ready
            self._prep_event = None
        else:
            self._backward_prep(ws, st)
            ws["scat_all"].zero_()
        self._pdl(False)
        det = self.deterministic
        check((lib.scann_rmse_prepare_det if det else lib.scann_rmse_prepare)(
            _p(ws["y"]), _p(target), b.B, _p(ws["dy"]), _p(self.grads, n), st), "rmse_prepare")
        self._pdl(True)
        self._ev("ga_backward", True)
        head = (_p(ws["head_slots"]), _p(ws["head_bslots"])) if det else \
            (self.gw("predict_property/kernel"), self.gw("predict_property/bias"))
        check((lib.scann_ga_head_backward_det if det else lib.scann_ga_head_backward)(
            _p(ws["qk"]), _p(b.atom_mask), b.B, b.M, int(sp.use_ga_norm), self.wT("bf_property/kernel"),
            self.w("predict_property/kernel"), _p(ws["tb"]), _p(ws["dy"]), _p(ws["d_qk"]), _p(ws["d_tb"]), *head, st),
              "ga_head_backward")
        self._ev("ga_backward", False)
        self.launches += 2
        if self.use_chain and self.tc_la_bwd:
            return self._backward_chained(b, ws, fork, wgrad, side, main, sst)
        dqk = ws["d_qk"]
        self._dense([_p(dqk), _p(dqk, D)], 2 * D,
                    [self.wT("global_attention/query/kernel"), self.wT("global_attention/key/kernel")], None, 2, 1, R,
                    _p(ws["d_ta"]), D, mode=2, pre_in=ws["ta"])
        dx = ws["dx"]
        self._dense([_p(ws["d_ta"])], D, [self.wT("after_Lc/kernel")], None, 1, 1, R, _p(dx), D)
        fork()
        wgrad([_p(ws["ctxg"])], D, [_p(ws["d_tb"])], D, 1, 1, b.B, [self.gw("bf_property/kernel")],
              [self.gw("bf_property/bias")])
        wgrad([_p(ws["xa"])], D, [_p(dqk), _p(dqk, D)], 2 * D, 1, 2, R,
              [self.gw("global_attention/query/kernel"), self.gw("global_attention/key/kernel")],
              [self.gw("global_attention/query/bias"), self.gw("global_attention/key/bias")])
        wgrad([_p(ws["x"][L])], D, [_p(ws["d_ta"])], D, 1, 1, R, [self.gw("after_Lc/kernel")], [self.gw("after_Lc/bias")])
        dg_up = None
        for l in range(L - 1, -1, -1):
            la = layer_name("local_attention", l)
            rn = layer_name("residual_norm", l)
            fg = f"{la}/filter_geo/kernel"
            d_v2, d_t1, dq = ws["d_v2"][l], ws["d_t1"][l], ws["dq"][l]
            if sp.use_attn_norm:
                check(lib.scann_layernorm_backward(_p(dx), _p(ws["v2"][l]), self.w(f"{rn}/layer_norm/gamma"), R,
                                                   _p(d_v2), 0, D, self.gw(f"{rn}/layer_norm/gamma"),
                                                   self.gw(f"{rn}/layer_norm/beta"), st), "ln_bwd")
                self._dense([_p(d_v2)], D, [self.wT(f"{rn}/dense_1/kernel")], None, 1, 1, R, _p(d_t1), D,
                            mode=2, pre_in=ws["t1"][l])
                self._dense([_p(d_t1)], D, [self.wT(f"{rn}/dense/kernel")], None, 1, 1, R, _p(ws["d_h"]), D,
                            resid=d_v2)
                d_h = ws["d_h"]
                self.launches += 1
            else:
                d_h = dx
            check(lib.scann_layernorm_backward(_p(d_h), _p(ws["ctxpre"][l]), self.w(f"{la}/layer_norm/gamma"), R,
                                               _p(ws["d_ctx"]), _p(dq), D, self.gw(f"{la}/layer_norm/gamma"),
                                               self.gw(f"{la}/layer_norm/beta"), st), "ln_bwd")
            scat = ws["scat"][l]
            s_pre, t_sc, dx_sc = scat[0], scat[1], scat[2]
            dg_out = ws["dg"][(L - l) % 2]
            self._ev("la_backward", True)
            if "la_bwd" in self._skip:
                pass
            elif self.tc_la_bwd:
                dg_buf = ws["dg"][(L - 1 - l) % 2]
                check(lib.scann_la_backward_tc(self.la_grid, b.stride, b.mma_rows, _p(b.ntiles), _p(b.tile_a0), _p(b.tile_a1), _p(b.cnt),
                                               _p(b.rowptr), _p(b.pair_c), _p(b.pair_j), _p(ws["x"][l]),
                                               _p(ws["proj"][l]), _p(ws["g"][l]), _p(ws["g"][l + 1]),
                                               _p(ws["kk"][l]), _p(ws["pre"][l]), self.wT(fg, D * D),
                                               self.wT(f"{la}/key/kernel"), self.w(f"{la}/layer_norm_g/gamma"),
                                               _p(ws["d_ctx"]), _p(dg_buf), int(dg_up is not None), _p(dg_out),
                                               _p(dq), _p(s_pre), _p(t_sc), _p(dx_sc), 0,
                                               self.gw(f"{la}/layer_norm_g/gamma"), self.gw(f"{la}/layer_norm_g/beta"),
                                               self.gw(f"{la}/key/bias"), *self._adrop(True, l), st), "la_backward_tc")
                self.launches += 2
            else:
                check(lib.scann_la_backward(self.la_grid, _p(b.ntiles), _p(b.tile_a0), _p(b.tile_a1), _p(b.cnt),
                                            _p(b.rowptr), _p(b.pair_c), _p(b.pair_j), _p(ws["x"][l]), _p(ws["proj"][l]),
                                            _p(ws["g"][l]), self.w(fg, D * D), self.w(f"{la}/key/kernel"),
                                            self.wT(fg, D * D), self.wT(f"{la}/key/kernel"), self.w(f"{la}/key/bias"),
                                            self.w(f"{la}/layer_norm_g/gamma"), self.w(f"{la}/layer_norm_g/beta"),
                                            _p(ws["d_ctx"]), _p(dg_up), _p(dg_out), _p(dq), _p(s_pre), _p(t_sc),
                                            _p(dx_sc), _p(ws["wpart"]),
                                            self.gw(f"{la}/layer_norm_g/gamma"), self.gw(f"{la}/layer_norm_g/beta"),
                                            self.gw(f"{la}/key/bias"), st), "la_backward")
                self.launches += 1
            self._ev("la_backward", False)
            # next link of the critical path: gradient w.r.t. the layer input x_l
            self._dense([_p(s_pre), _p(t_sc), _p(dq)], D,
                        [self.wT(fg, 0), self.wT(fg, 2 * D * D), self.wT(f"{la}/query/kernel")], None, 3, 1, R, _p(dx),
                        D, resid=dx_sc)
            # ---- weight gradients of this layer (side stream)
            if "wgrad" in self._skip:
                dg_up = dg_out
                continue
            fork()
            if self.tc_la_bwd:
                check(lib.scann_la_wgrad_tc(self.la_grid, b.stride, _p(b.ntiles), _p(b.pair_c), _p(b.pair_j), _p(ws["x"][l]),
                                            _p(ws["g"][l]), _p(ws["g"][l + 1]), _p(ws["kk"][l]), _p(ws["pre"][l]),
                                            _p(ws["wpart"]), sst), "la_wgrad_tc")
                self.launches += 2
            check(lib.scann_la_wpart_reduce(_p(ws["wpart"]), _p(b.ntiles), self.la_grid, b.stride, self.gw(f"{la}/key/kernel"),
                                            self.gw(fg, D * D), sst), "la_wpart_reduce")
            self.launches += 1
            if sp.use_attn_norm:
                wgrad([_p(ws["h1"][l])], D, [_p(d_v2)], D, 1, 1, R, [self.gw(f"{rn}/dense_1/kernel")],
                      [self.gw(f"{rn}/dense_1/bias")])
                wgrad([_p(ws["h"][l])], D, [_p(d_t1)], D, 1, 1, R, [self.gw(f"{rn}/dense/kernel")],
                      [self.gw(f"{rn}/dense/bias")])
            wgrad([_p(ws["x"][l])], D, [_p(s_pre), _p(t_sc), _p(dq)], D, 1, 3, R,
                  [self.gw(fg, 0), self.gw(fg, 2 * D * D), self.gw(f"{la}/query/kernel")],
                  [self.gw(f"{la}/filter_geo/bias"), 0, self.gw(f"{la}/query/bias")])
            dg_up = dg_out
        self._backward_tail(b, ws, dg_up, side, main)

    def _backward_tail(self, b: Batch, ws: dict, dg_up, side, main) -> None:
        """Geometry-initialisation and embedding backward, then the join with the weight-gradient stream."""
        sp, st = self.spec, self._stream()
        R = b.R
        dx = ws["dx"]
        self._pdl(False)
        if sp.g_update and "geom_init" not in self._skip:
            # geometry-initialisation backward (a full-grid FP32 kernel, ~25 us) and the embedding backward (two small
            # latency-bound launches, ~17 us) only meet in the optimiser: the former goes to the side stream
            gst = st
            if side is not main and self.tail_fork:
                ev = torch.cuda.Event()
                ev.record(main)
                side.wait_event(ev)
                gst = side.cuda_stream
            if self.deterministic:
                check(lib.scann_geom_init_backward_det(
                    _p(b.ntiles), self.la_grid * self.gi_bwd_mult, b.stride, _p(b.pair_c), _p(b.pair_d), _p(b.pair_w),
                    _p(self.centers_d), _p(self.centers_w), self.w("neighbor_d/kernel"), self.w("neighbor_d/bias"),
                    self.w("neighbor_w/kernel"), self.w("neighbor_w/bias"), _p(dg_up), _p(ws["gi_slots"]), gst),
                      "geom_init_backward_det")
            else:
                check(lib.scann_geom_init_backward(_p(b.ntiles), self.la_grid * self.gi_bwd_mult, b.stride, _p(b.pair_c), _p(b.pair_d), _p(b.pair_w),
                                                   _p(self.centers_d), _p(self.centers_w), self.w("neighbor_d/kernel"),
                                                   self.w("neighbor_d/bias"), self.w("neighbor_w/kernel"),
                                                   self.w("neighbor_w/bias"), _p(dg_up), self.gw("neighbor_d/kernel"),
                                                   self.gw("neighbor_d/bias"), self.gw("neighbor_w/kernel"),
                                                   self.gw("neighbor_w/bias"), gst), "geom_init_backward")
        E = sp.embedding_dim
        ring = sp.use_ring
        if sp.feature == "cgcnn" and b.route != TABLE_ROUTE:
            # deterministic mode: dense_embed's gradients go to per-CTA slots (scann_slot_reduce)
            dense = (_p(ws["cg_slots"]),) if self.deterministic else \
                (self.gw("dense_embed/kernel"), self.gw("dense_embed/bias"))
            check((lib.scann_cgcnn_embed_backward_det if self.deterministic else lib.scann_cgcnn_embed_backward)(
                _p(b.atomic92), _p(ws["emb_rows"]), _p(b.ring) if ring else 0, R, 92, E,
                self.w("extra_embed/kernel") if ring else 0, self.w("extra_embed/bias") if ring else 0,
                self.w("dense_embed/kernel"), _p(ws["t0"]), _p(dx), _p(ws["d_cat"]), self.gw("embed_atom/kernel"),
                self.gw("embed_atom/bias"), self.gw("extra_embed/kernel") if ring else 0,
                self.gw("extra_embed/bias") if ring else 0, *dense, _p(self.adam_scalars, 8), st), "cgcnn_embed_backward")
            self.launches += 2
            if side is not main:
                ev = torch.cuda.Event()
                ev.record(side)
                main.wait_event(ev)
            return
        if b.route == TABLE_ROUTE:
            # the per-element gradient of emb_table lands in the zeroed d_emb, then goes through the table into
            # embed_atom's kernel / bias (scann_cgcnn_table_backward)
            tab = self._tab
            n_emb, emb, G, d_emb = self.atomic_features.shape[0], _p(tab["emb"]), tab["G"], _p(tab["d_emb"])
            tab["d_emb"].zero_()
            if self.deterministic:
                ns = lib.scann_embed_backward_det_slots(R)
                if ws.get("emb_slots_table") is None or ws["emb_slots_table"].shape[:2] != (ns, n_emb + 3):
                    ws["emb_slots_table"] = torch.empty(ns, n_emb + 3, D, dtype=torch.float32, device=self.device)
                Gslots = (_p(ws["emb_slots_table"]),)
            else:
                Gslots = ()
        else:
            n_emb, emb, G, d_emb = sp.n_atoms, self.w("embed_atom/embeddings"), ws["G"], self.gw("embed_atom/embeddings")
            Gslots = (_p(ws["emb_slots"]),) if self.deterministic else ()
        check((lib.scann_embed_backward_det if self.deterministic else lib.scann_embed_backward)(
            _p(b.atomic), _p(b.ring) if ring else 0, R, E, n_emb, emb,
            self.w("extra_embed/kernel") if ring else 0, self.w("extra_embed/bias") if ring else 0,
            self.w("dense_embed/kernel"), _p(ws["t0"]), _p(dx), _p(G), *Gslots,
            d_emb, self.gw("extra_embed/kernel") if ring else 0,
            self.gw("extra_embed/bias") if ring else 0, self.gw("dense_embed/kernel"), self.gw("dense_embed/bias"),
            _p(self.adam_scalars, 8), st), "embed_backward")
        self.launches += 4
        if b.route == TABLE_ROUTE:
            check(lib.scann_cgcnn_table_backward(_p(self.atomic_features), d_emb, n_emb, 92, E, self.gw("embed_atom/kernel"),
                                                 self.gw("embed_atom/bias"), st), "cgcnn_table_backward")
            self.launches += 1
        if side is not main:             # join: the optimiser needs every weight gradient
            ev = torch.cuda.Event()
            ev.record(side)
            main.wait_event(ev)

    def _backward_chained(self, b: Batch, ws: dict, fork, wgrad, side, main, sst) -> None:
        """Backward layers with the per-atom links fused (scann_dense_chain):
        [GA projections^T, after_Lc^T, tail(L-1)] -> LA_bwd(L-1) -> [x-gradient of layer L-1, tail(L-2)] -> ... ->
        LA_bwd(0) -> [x-gradient of layer 0] -> geometry init / embedding backward.
        tail(l) turns the gradient w.r.t. x_{l+1} into d_ctx / dq of layer l: LayerNorm backward of ResidualNorm,
        its two Dense layers transposed (swish'), LayerNorm backward of the attention output."""
        sp, st = self.spec, self._stream()
        L, R = sp.n_attention, b.R
        dqk, dx = ws["d_qk"], ws["dx"]

        def with_tail(head: dict, l: int):
            """``head``: keyword arguments of the GEMM step that produces d x_{l+1}; returns the step list."""
            la = layer_name("local_attention", l)
            rn = layer_name("residual_norm", l)
            la_ln = dict(mode=4, pre_in=_p(ws["ctxpre"][l]), gamma=self.w(f"{la}/layer_norm/gamma"),
                         **self._ln_grads(ws, l, 0, la), C_=_p(ws["d_ctx"]), C2=_p(ws["dq"][l]))
            if not sp.use_attn_norm:
                return [chain_step(**head, **la_ln)]
            d_v2, d_t1 = ws["d_v2"][l], ws["d_t1"][l]
            return [
                # d_v2 (residual branch) and d_v2 * dropout mask (gradient of the dense_1 output, also the operand
                # of the next step and of the dense_1 weight gradient)
                chain_step(**head, mode=4, pre_in=_p(ws["v2"][l]), gamma=self.w(f"{rn}/layer_norm/gamma"),
                           **self._ln_grads(ws, l, 1, rn), C_=_p(d_v2), C2=_p(ws["d_v2m"][l]), to_image=True,
                           drop=_p(self.adam_scalars, 8), drop_site=1 + l),
                chain_step(W=[self.wT(f"{rn}/dense_1/kernel")], mode=2, pre_in=_p(ws["t1"][l]), C_=_p(d_t1), to_image=True),
                chain_step(W=[self.wT(f"{rn}/dense/kernel")], resid=_p(d_v2), **la_ln),
            ]

        steps = [chain_step(A=[_p(dqk), _p(dqk, D)], lda=2 * D,
                            W=[self.wT("global_attention/query/kernel"), self.wT("global_attention/key/kernel")],
                            mode=2, pre_in=_p(ws["ta"]), C_=_p(ws["d_ta"]), to_image=True)]
        steps += with_tail(dict(W=[self.wT("after_Lc/kernel")]), L - 1)
        self._chain(steps, R)
        batched = self.use_wgrad_batch
        if not batched:
            fork()
            wgrad([_p(ws["ctxg"])], D, [_p(ws["d_tb"])], D, 1, 1, b.B, [self.gw("bf_property/kernel")],
                  [self.gw("bf_property/bias")])
            wgrad([_p(ws["xa"])], D, [_p(dqk), _p(dqk, D)], 2 * D, 1, 2, R,
                  [self.gw("global_attention/query/kernel"), self.gw("global_attention/key/kernel")],
                  [self.gw("global_attention/query/bias"), self.gw("global_attention/key/bias")])
            wgrad([_p(ws["x"][L])], D, [_p(ws["d_ta"])], D, 1, 1, R, [self.gw("after_Lc/kernel")],
                  [self.gw("after_Lc/bias")])
        dg_up = None
        for l in range(L - 1, -1, -1):
            la = layer_name("local_attention", l)
            rn = layer_name("residual_norm", l)
            fg = f"{la}/filter_geo/kernel"
            d_v2, d_t1, dq = ws["d_v2"][l], ws["d_t1"][l], ws["dq"][l]
            scat = ws["scat"][l]
            s_pre, t_sc, dx_sc = scat[0], scat[1], scat[2]
            dg_out = ws["dg"][(L - l) % 2]
            dg_buf = ws["dg"][(L - 1 - l) % 2]
            self._ev("la_backward", True)
            if not sp.g_update:
                # SCANN without geometry update: attention part only, then the filter_geo [20,128] gradient
                if self.deterministic:
                    # d_a * g' stored per pair, summed per atom row in list order behind the filter gradient
                    check(lib.scann_la_backward_pipe_det(
                        self.la_grid, b.rows, 1, _p(b.ntiles), _p(b.pair_c), _p(b.pair_j), _p(ws["x"][l]), _p(ws["proj"][l]),
                        0, _p(ws["gsave"][l]), _p(ws["kk"][l]), 0, 0, self.wT(f"{la}/key/kernel"), 0, _p(ws["d_ctx"]),
                        _p(ws["dg"][0]), 0, 0, _p(dq), 0, 0, _p(ws["pairbuf"]), 0, 0, _p(ws["dbk_slots"][l]),
                        *self._adrop(True, l), _p(self.status), st), "la_backward_pipe_det")
                elif self.noup_pipe and b.stride == 32:
                    check(lib.scann_la_backward_pipe(
                        self.la_grid, b.rows, 1, _p(b.ntiles), _p(b.pair_c), _p(b.pair_j), _p(ws["x"][l]), _p(ws["proj"][l]),
                        0, _p(ws["gsave"][l]), _p(ws["kk"][l]), 0, 0, self.wT(f"{la}/key/kernel"), 0, _p(ws["d_ctx"]),
                        _p(ws["dg"][0]), 0, 0, _p(dq), 0, 0, _p(dx_sc), 0, 0, self.gw(f"{la}/key/bias"),
                        *self._adrop(True, l), _p(self.status), st), "la_backward_pipe")
                else:
                    check(lib.scann_la_backward_noupdate_tc(
                        self.la_grid, b.stride, b.mma_rows, _p(b.ntiles), _p(b.tile_a0), _p(b.tile_a1), _p(b.cnt), _p(b.rowptr),
                        _p(b.pair_c), _p(b.pair_j), _p(ws["x"][l]), _p(ws["proj"][l]), _p(ws["gsave"][l]), _p(ws["kk"][l]),
                        self.wT(f"{la}/key/kernel"), _p(ws["d_ctx"]), _p(ws["dg"][0]), _p(dq), _p(dx_sc),
                        self.gw(f"{la}/key/bias"), *self._adrop(True, l), st), "la_backward_noupdate_tc")
                if self.deterministic:
                    check(lib.scann_noupdate_geom_backward_det(
                        _p(b.ntiles), self.la_grid * self.gi_bwd_mult, b.stride, _p(b.pair_c), _p(b.pair_d), _p(b.pair_w),
                        _p(self.centers_d), self.w(fg), self.w(f"{la}/filter_geo/bias"), _p(ws["dg"][0]),
                        _p(ws["noup_slots"][l]), st), "noupdate_geom_backward_det")
                    check(lib.scann_row_gather(R, _p(b.inv_ptr), _p(b.inv_idx), _p(ws["pairbuf"]), _p(dx_sc), 0, 0, st),
                          "row_gather")
                    self.launches += 1
                else:
                    check(lib.scann_noupdate_geom_backward(
                        _p(b.ntiles), self.la_grid * self.gi_bwd_mult, b.stride, _p(b.pair_c), _p(b.pair_d), _p(b.pair_w), _p(self.centers_d),
                        self.w(fg), self.w(f"{la}/filter_geo/bias"), _p(ws["dg"][0]), self.gw(fg),
                        self.gw(f"{la}/filter_geo/bias"), st), "noupdate_geom_backward")
                self.launches += 2
            elif "la_bwd" not in self._skip:
                plan_args = (_p(b.ntiles), _p(b.tile_a0), _p(b.tile_a1), _p(b.cnt), _p(b.rowptr), _p(b.pair_c), _p(b.pair_j))
                data = (_p(ws["x"][l]), _p(ws["proj"][l]), _p(ws["g"][l]), _p(ws["g"][l + 1]), _p(ws["kk"][l]),
                        _p(ws["pre"][l]), self.wT(fg, D * D), self.wT(f"{la}/key/kernel"),
                        self.w(f"{la}/layer_norm_g/gamma"), _p(ws["d_ctx"]), _p(dg_buf), int(dg_up is not None),
                        _p(dg_out), _p(dq), _p(s_pre), _p(t_sc), _p(dx_sc))
                grads = (self.gw(f"{la}/layer_norm_g/gamma"), self.gw(f"{la}/layer_norm_g/beta"), self.gw(f"{la}/key/bias"))
                pipe = (self.la_pipe >> 2) & 3 if b.stride == 32 else 0
                if self.deterministic:
                    # d_a * g' stored per pair, d_pre left per pair in pre[l]; both summed per atom row in list order
                    data = data[:-1] + (_p(ws["pairbuf"]),)
                    grads = (_p(ws["lng_slots"][l]), 0, _p(ws["dbk_slots"][l]))
                    check(lib.scann_la_backward_pipe_det(self.la_grid, b.rows, 3, plan_args[0], plan_args[5], plan_args[6],
                                                         *data, *grads, *self._adrop(True, l), _p(self.status), st),
                          "la_backward_pipe_det")
                    check(lib.scann_row_gather(R, _p(b.inv_ptr), _p(b.inv_idx), _p(ws["pairbuf"]), _p(dx_sc),
                                               _p(ws["pre"][l]), _p(t_sc), st), "row_gather")
                    pipe = 0
                    self.launches += 1
                for part in ((1, 2) if not self.deterministic else ()):   # attention kernel, then geometry kernel
                    if pipe & part:
                        check(lib.scann_la_backward_pipe(self.la_grid, b.rows, part, plan_args[0], plan_args[5], plan_args[6],
                                                         *data, *grads, *self._adrop(True, l), _p(self.status), st),
                              "la_backward_pipe")
                    else:
                        check(lib.scann_la_backward_tc_part(part, self.la_grid, b.stride, b.mma_rows, *plan_args, *data, 0,
                                                            *grads, *self._adrop(True, l), st), "la_backward_tc")
                self.launches += 2
            self._ev("la_backward", False)
            # next link of the critical path: gradient w.r.t. the layer input x_l, then the tail of layer l-1
            if sp.g_update:
                head = dict(A=[_p(s_pre), _p(t_sc), _p(dq)], W=[self.wT(fg, 0), self.wT(fg, 2 * D * D),
                                                               self.wT(f"{la}/query/kernel")], resid=_p(dx_sc))
            else:
                head = dict(A=[_p(dq)], W=[self.wT(f"{la}/query/kernel")], resid=_p(dx_sc))
            self._chain(with_tail(head, l - 1) if l > 0 else [chain_step(**head, C_=_p(dx))], R)
            dg_up = dg_out
            # ---- weight gradients of this layer (side stream), unless they are batched at the end
            if "wgrad" in self._skip or batched:
                continue
            fork()
            check(lib.scann_la_wgrad_tc(self.la_grid, b.stride, _p(b.ntiles), _p(b.pair_c), _p(b.pair_j), _p(ws["x"][l]),
                                        _p(ws["g"][l]), _p(ws["g"][l + 1]), _p(ws["kk"][l]), _p(ws["pre"][l]),
                                        _p(ws["wpart"]), sst), "la_wgrad_tc")
            check(lib.scann_la_wpart_reduce(_p(ws["wpart"]), _p(b.ntiles), self.la_grid, b.stride,
                                            self.gw(f"{la}/key/kernel"), self.gw(fg, D * D), sst), "la_wpart_reduce")
            self.launches += 3
            if sp.use_attn_norm:
                wgrad([_p(ws["h1"][l])], D, [_p(ws["d_v2m"][l])], D, 1, 1, R, [self.gw(f"{rn}/dense_1/kernel")],
                      [self.gw(f"{rn}/dense_1/bias")])
                wgrad([_p(ws["h"][l])], D, [_p(d_t1)], D, 1, 1, R, [self.gw(f"{rn}/dense/kernel")],
                      [self.gw(f"{rn}/dense/bias")])
            wgrad([_p(ws["x"][l])], D, [_p(s_pre), _p(t_sc), _p(dq)], D, 1, 3, R,
                  [self.gw(fg, 0), self.gw(fg, 2 * D * D), self.gw(f"{la}/query/kernel")],
                  [self.gw(f"{la}/filter_geo/bias"), 0, self.gw(f"{la}/query/bias")])
        if batched and "wgrad" not in self._skip:
            self._pdl(False)
            self._ev("wgrad_batch", True)
            # deterministic mode: each launch's reduce has read the slots before the next launch (same stream) rewrites them
            for table, count in self._wgrad_table(b, ws):
                if self.deterministic:
                    check(lib.scann_wgrad_batch_tc_det(self.la_grid, table, count, _p(b.ntiles), b.stride, _p(b.pair_c),
                                                       _p(b.pair_j), _p(b.valid_rows), _p(b.valid_j), _p(b.nvalid),
                                                       _p(ws["wg_slots"]), _p(ws["wg_bslots"]), st), "wgrad_batch_tc_det")
                    check(lib.scann_wgrad_batch_reduce(self.la_grid, table, count, _p(b.ntiles), b.stride,
                                                       _p(b.valid_rows), _p(b.nvalid), _p(ws["wg_slots"]),
                                                       _p(ws["wg_bslots"]), st), "wgrad_batch_reduce")
                    self.launches += 1
                else:
                    check(lib.scann_wgrad_batch_tc(self.la_grid, table, count, _p(b.ntiles), b.stride, _p(b.pair_c),
                                                   _p(b.pair_j), _p(b.valid_rows), _p(b.valid_j), _p(b.nvalid), st),
                          "wgrad_batch_tc")
                self.launches += 1
            self._ev("wgrad_batch", False)
        self._backward_tail(b, ws, dg_up, side, main)

    def _wgrad_table(self, b: Batch, ws: dict):
        """Device table of all dW += X^T Y problems of a train step (pointers into this workspace), as the
        (device address, problem count) of each launch: 4 + 7 L problems for SCANN+ with attention normalisation, at most
        scann_wgrad_batch_max_problems() per launch (one launch up to 13 layers)."""
        if "wg_launches" in ws:
            return ws["wg_launches"]
        sp = self.spec
        L, R = sp.n_attention, b.R
        probs = []

        def add(X, Y, dW, db=0, xg=0, ldx=D, ldy=D, rows=R):
            pr = WgradProblem()
            pr.X, pr.Y, pr.xg, pr.dW, pr.db = X or None, Y or None, xg or None, dW or None, db or None
            pr.ldx, pr.ldy, pr.rows, pr.pad = ldx, ldy, rows, 0
            probs.append(pr)

        dqk = ws["d_qk"]
        add(_p(ws["ctxg"]), _p(ws["d_tb"]), self.gw("bf_property/kernel"), self.gw("bf_property/bias"), rows=b.B)
        add(_p(ws["xa"]), _p(dqk), self.gw("global_attention/query/kernel"), self.gw("global_attention/query/bias"),
            ldy=2 * D)
        add(_p(ws["xa"]), _p(dqk, D), self.gw("global_attention/key/kernel"), self.gw("global_attention/key/bias"),
            ldy=2 * D)
        add(_p(ws["x"][L]), _p(ws["d_ta"]), self.gw("after_Lc/kernel"), self.gw("after_Lc/bias"))
        for l in range(L - 1, -1, -1):
            la = layer_name("local_attention", l)
            rn = layer_name("residual_norm", l)
            fg = f"{la}/filter_geo/kernel"
            scat = ws["scat"][l]
            if sp.g_update:
                add(_p(ws["g"][l + 1]), _p(ws["kk"][l]), self.gw(f"{la}/key/kernel"), xg=_p(ws["x"][l]), rows=-1)
                add(_p(ws["g"][l]), _p(ws["pre"][l]), self.gw(fg, D * D), rows=-1)
            else:
                add(_p(ws["gsave"][l]), _p(ws["kk"][l]), self.gw(f"{la}/key/kernel"), xg=_p(ws["x"][l]), rows=-1)
            if sp.use_attn_norm:
                add(_p(ws["h1"][l]), _p(ws["d_v2m"][l]), self.gw(f"{rn}/dense_1/kernel"), self.gw(f"{rn}/dense_1/bias"))
                add(_p(ws["h"][l]), _p(ws["d_t1"][l]), self.gw(f"{rn}/dense/kernel"), self.gw(f"{rn}/dense/bias"))
            if sp.g_update:
                add(_p(ws["x"][l]), _p(scat[0]), self.gw(fg, 0), self.gw(f"{la}/filter_geo/bias"))
                add(_p(ws["x"][l]), _p(scat[1]), self.gw(fg, 2 * D * D))
            add(_p(ws["x"][l]), _p(ws["dq"][l]), self.gw(f"{la}/query/kernel"), self.gw(f"{la}/query/bias"))
        arr = (WgradProblem * len(probs))(*probs)
        host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
        ws["wg_table"] = host.to(self.device)
        step, size = lib.scann_wgrad_batch_max_problems(), ctypes.sizeof(WgradProblem)
        ws["wg_launches"] = [(_p(ws["wg_table"], i * size), min(step, len(probs) - i)) for i in range(0, len(probs), step)]
        return ws["wg_launches"]

    def _backward_prep(self, ws: dict, stream: int) -> None:
        """Work the backward needs that does not depend on the forward: transposed weight blocks and
        zeroed scatter targets."""
        check(lib.scann_transpose_blocks(_p(self.params), _p(self.paramsT), _p(self.tblocks), self.tblocks.numel(),
                                         stream), "transpose_blocks")
        self.launches += 1

    # ------------------------------------------------------------------ optimiser
    def _set_adam(self, lr: float, batch_global: int, decay: float = 1e-5, b1=0.9, b2=0.999, eps=1e-7):
        t = self.step_count + 1
        lr_t = lr / (1.0 + decay * (t - 1))                       # legacy Keras `decay`
        alpha = lr_t * np.sqrt(1.0 - b2 ** t) / (1.0 - b1 ** t)
        h = self._adam_host
        if self._adam_ev is not None:
            self._adam_ev.synchronize()
        h[0], h[1], h[2], h[3], h[4], h[5] = alpha, b1, b2, eps, L2_COEF, float(batch_global)
        hi = h.numpy().view(np.uint32)
        self.last_drop_seed = (self.dropout_seed * 2654435761 + 40503 * t) & 0xFFFFFFFF
        hi[8] = self.last_drop_seed
        hi[9] = min(int(self.dropout_rate * 4294967296.0), 0xFFFFFFFF)
        hi[10] = np.float32(1.0 / (1.0 - self.dropout_rate)).view(np.uint32)
        hi[11] = 1 if self.train_dropout else 0
        hi[12] = self.last_drop_seed                       # attention-probability Dropout (use_drop): rate 0.05
        hi[13] = min(int(0.05 * 4294967296.0), 0xFFFFFFFF)
        hi[14] = np.float32(1.0 / (1.0 - 0.05)).view(np.uint32)
        hi[15] = 1 if (self.train_dropout and self.spec.use_drop) else 0
        self.adam_scalars.copy_(h, non_blocking=True)
        self._adam_ev = torch.cuda.Event()
        self._adam_ev.record(torch.cuda.current_stream(self.device))

    def loss_value(self, batch_global: int) -> torch.Tensor:
        """[loss (RMSE + l2 terms), RMSE, MAE] of the batch whose SSE sits in the gradient arena."""
        n = self.layout.total
        sse = _p(self.p2p.sums) if self.p2p is not None else _p(self.grads, n)
        check(lib.scann_loss_value(_p(self.params), _p(self.l2mask), n, sse, float(batch_global),
                                   L2_COEF, _p(self.loss_out), self._stream()), "loss_value")
        self.launches += 1
        return self.loss_out

    def loss_value_async(self, batch_global: int, slots: int = 8):
        """``loss_value`` followed by an asynchronous device->host copy into a ring of pinned slots: returns
        ``(pinned tensor, event)``; the values are valid once the event has completed.  A slot is reused after
        ``slots`` further calls (read it before)."""
        lv = self.loss_value(batch_global)
        if len(self._loss_ring) < slots:
            self._loss_ring.append(torch.zeros(4, dtype=torch.float32).pin_memory())
        self._loss_pos = (getattr(self, "_loss_pos", -1) + 1) % slots
        pin = self._loss_ring[self._loss_pos]
        pin.copy_(lv, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        return pin, ev

    def train_step(self, b: Batch, target, lr: float, allreduce=None, batch_global: Optional[int] = None,
                   apply: bool = True, want_grads: bool = False, replan: bool = False) -> None:
        """One Keras train_step (scann_model.py:232-241): forward, RMSE + l2 loss, backward, Adam.
        ``allreduce(tensor)`` sums the gradient arena (+SSE) across data-parallel ranks.  With
        ``replan`` the pair plan is rebuilt from the (freshly loaded) inputs as part of the step.
        The kernel sequence of a shape class is captured once into a CUDA graph and replayed."""
        if target is not None and target is not b.target:
            self.set_target(b, target)
        if self.train_dropout and not (self.use_chain and self.tc_la_bwd):
            raise NotImplementedError("training-mode Dropout needs the chained tensor-core engine (SCANN_CHAIN=1)")
        self._set_adam(lr, batch_global or b.B)
        self._flush_host(b)
        key = ("train", replan, apply, want_grads, allreduce is not None)
        if b.route:
            key += (b.route,)
        if not self.use_graphs or self.prof is not None:
            self._train_body(b, allreduce, apply, want_grads, replan)
        else:
            g = b.graphs.get(key)
            if g is None:
                # one eager pass allocates workspaces / warms up, then capture on a side stream.  With the peer-memory
                # exchange the pass stays local (it applies nothing): ranks that meet a new batch shape at different
                # steps would otherwise disagree on the number of exchanges
                self._train_body(b, allreduce, apply=False, want_grads=False, replan=replan, exchange=False)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                n0 = self.launches
                with torch.cuda.graph(g):
                    self._train_body(b, allreduce, apply, want_grads, replan)
                g.n_launches = self.launches - n0
                b.graphs[key] = g
                self.graph_captures += 1
            else:
                self.launches += g.n_launches
            g.replay()
        if apply:
            self.step_count += 1
            self._wimg_dirty = True      # the parameters moved: the next forward rebuilds the weight operand images

    def _train_body(self, b: Batch, allreduce, apply: bool, want_grads: bool, replan: bool, exchange: bool = True) -> None:
        p2p = self.p2p if exchange else None
        if self.deterministic:
            self._check_deterministic_support()
            self._check_deterministic_batch(b)
            if allreduce is not None and not self._nccl_warned:
                import warnings
                warnings.warn("deterministic mode: the cross-rank gradient sum of the NCCL all-reduce runs in NCCL's "
                              "order, which this package does not control", RuntimeWarning)
                self._nccl_warned = True
        if self.p2p is not None:
            # no peer still reads the arena that is zeroed next (scann_b200/csrc/p2p.cu); also in the local warm pass
            check(lib.scann_p2p_begin_step(_p(self.p2p.block), _p(self.p2p.sums), self._stream()), "p2p_begin_step")
            self.launches += 1
        self.grads.zero_()
        ws = self._workspace(b, True)

        def prep():
            # overlaps with the forward (side stream, behind the embedding): weight transposes and the zero-fill of
            # the scatter targets of the backward pass
            if self.use_side_stream:
                self._backward_prep(ws, self.side_stream.cuda_stream)
                ws["scat_all"].zero_()
                self._prep_event = torch.cuda.Event()
                self._prep_event.record(self.side_stream)

        self.forward(b, training=True, replan=replan, side_work=prep)
        self.backward(b, b.target)
        n = self.layout.total
        if self.deterministic:
            self._pdl(False)
            sfx = "_" + b.route if b.route else ""
            check(lib.scann_slot_reduce(_p(ws["slot_table" + sfx]), ws["slot_count" + sfx], ws["slot_max"],
                                        self._stream()), "slot_reduce")
            self.launches += 1
        if p2p is not None:
            if self.deterministic:
                check(lib.scann_adam_p2p_step_det(_p(self.params), _p(self.adam_m), _p(self.adam_v), _p(self.l2mask), n,
                                                  _p(self.p2p.block), _p(self.p2p.sums), _p(self.adam_scalars),
                                                  _p(self.grad_out) if want_grads else 0, int(apply), _p(ws["reg_slots"]),
                                                  self._stream()), "adam_p2p_step_det")
            else:
                check(lib.scann_adam_p2p_step(_p(self.params), _p(self.adam_m), _p(self.adam_v), _p(self.l2mask), n,
                                              _p(self.p2p.block), _p(self.p2p.sums), _p(self.adam_scalars),
                                              _p(self.grad_out) if want_grads else 0, int(apply), self._stream()),
                      "adam_p2p_step")
            self.launches += 1
            return
        if allreduce is not None and exchange:
            # (not in the local warm-up pass of a new shape class, whose result is discarded: ranks that meet new
            # shapes at different steps must still issue the same number of collectives)
            allreduce(self.grads)
        if self.deterministic:
            check(lib.scann_adam_step_det(_p(self.params), _p(self.grads), _p(self.adam_m), _p(self.adam_v), _p(self.l2mask),
                                          n, _p(self.grads, n), _p(self.adam_scalars),
                                          _p(self.grad_out) if want_grads else 0, int(apply), _p(ws["reg_slots"]),
                                          self._stream()), "adam_step_det")
            self.launches += 1
        else:
            check(lib.scann_adam_step(_p(self.params), _p(self.grads), _p(self.adam_m), _p(self.adam_v), _p(self.l2mask), n,
                                      _p(self.grads, n), _p(self.adam_scalars), _p(self.grad_out) if want_grads else 0,
                                      int(apply), self._stream()), "adam_step")
        self.launches += 1

    def predict_step(self, b: Batch, replan: bool = False, local_attention=False):
        """Inference forward (plan + graph of kernels) -> (y[B], ga[B*M]) device tensors.

        ``local_attention``: also return every layer's local-attention scores, ``(y, ga, scores)``.  The kernels store
        them in plan order and one more launch unpacks them (``_unpack_scores``); the graph that does so is captured
        under its own key, ``("infer", replan, layout)``, so the graph without scores stays as it is.  True or
        ``"padded"``: scores [L, B, 8, M, N], the reference's layout.  ``"csr"``: scores [L, 8, rows] whose first P
        columns are the batch's P pairs in the order of its CSR neighbour lists (lists without the padding marker
        1000, as ``voronoi.NeighborSelection.csr`` writes them).  The tensors belong to the shape class: the next step
        of the class overwrites them."""
        layout = score_layout(local_attention)
        key = ("infer", replan) if layout is None else ("infer", replan, layout)
        if b.route:
            key += (b.route,)
        self._flush_host(b)
        if self._wimg_dirty:
            self._weight_images()        # outside the captured graph: only needed after the parameters changed
        if layout is not None:
            self._score_buffers(b, layout)
        if not self.use_graphs or self.prof is not None:
            self._infer_body(b, replan, layout)
        else:
            g = b.graphs.get(key)
            if g is None:
                self._infer_body(b, replan, layout)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                n0 = self.launches
                with torch.cuda.graph(g):
                    self._infer_body(b, replan, layout)
                g.n_launches = self.launches - n0
                b.graphs[key] = g
                self.graph_captures += 1
            else:
                self.launches += g.n_launches
            g.replay()
        ws = self._workspace(b, False)
        if layout is None:
            return ws["y"], ws["ga"]
        return ws["y"], ws["ga"], b.scores[layout]

    def _infer_body(self, b: Batch, replan: bool, layout: Optional[str]) -> None:
        self.forward(b, training=False, attn=b.attn if layout is not None else None, replan=replan)
        if layout is not None:
            self._unpack_scores(b, layout)

    def _score_buffers(self, b: Batch, layout: str) -> None:
        """The shape class's buffers of the local-attention scores (allocated when first requested)."""
        L, dev = self.spec.n_attention, self.device
        if b.attn is None:
            b.attn = torch.empty(L, b.rows, 8, dtype=torch.float32, device=dev)
        if layout not in b.scores:
            shape = (L, b.B, 8, b.M, b.N) if layout == "padded" else (L, 8, b.rows)
            b.scores[layout] = torch.empty(shape, dtype=torch.float32, device=dev)

    def _unpack_scores(self, b: Batch, layout: str) -> None:
        """Plan-ordered scores (b.attn) -> b.scores[layout], one launch for all layers."""
        L, st = self.spec.n_attention, self._stream()
        self._ev("attn_unpack", True)
        if layout == "padded":
            check(lib.scann_attn_to_padded(_p(b.attn), L, b.rows, _p(b.cnt), _p(b.rowptr), _p(b.nmask), b.B, b.M, b.N,
                                           _p(b.scores[layout]), st), "attn_to_padded")
        else:
            check(lib.scann_attn_to_csr(_p(b.attn), L, b.rows, _p(b.valid_rows), _p(b.nvalid), b.rows,
                                        _p(b.scores[layout]), st), "attn_to_csr")
        self._ev("attn_unpack", False)
        self.launches += 1


def score_layout(local_attention) -> Optional[str]:
    """``local_attention`` argument of ``Engine.predict_step`` -> None, "padded" or "csr"."""
    if isinstance(local_attention, str):
        if local_attention not in ("padded", "csr"):
            raise ValueError(f"local_attention must be a bool, 'padded' or 'csr', not {local_attention!r}")
        return local_attention
    if not isinstance(local_attention, (bool, np.bool_)):
        raise TypeError(f"local_attention must be a bool, 'padded' or 'csr', not {type(local_attention).__name__}")
    return "padded" if local_attention else None
