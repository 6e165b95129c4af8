"""Local-attention scores of every layer: ``predict(..., local_attention=True)`` and
``predict_structures(..., local_attention=True)`` (``Engine.predict_step(local_attention=...)``, ``scann_attn_to_padded``
/ ``scann_attn_to_csr`` in csrc/plan.cu).

The reference returns them as the first output of each ``LocalAttention.call`` (attn[B,H,M,N],
scann/layers/attention.py:186-189, :216): the softmax over an atom's neighbour slots, 0 on masked slots and 1/N on rows
without a valid slot (in fp32 the mask's -1e9 absorbs every logit).  They are compared with the oracle's per-layer
``trace["attn{l}"]``."""
import numpy as np
import pytest

from tests.test_predict_structures import _model, host_iterator, hub, lone_atom, qm9_like


# ------------------------------------------------------------------------------------------------ CPU
def test_split_pair_scores_per_structure():
    from scann_b200.model import LocalAttentionScores, split_pair_scores
    sa = np.array([0, 2, 3, 6], np.int32)                 # 3 structures: 2, 1 and 3 atoms
    an = np.array([0, 3, 5, 5, 7, 8, 10], np.int32)       # atom 2 (structure 1) has no neighbour
    P, L = int(an[-1]), 2
    idx = np.arange(P, dtype=np.int32) % 3
    d = np.linspace(1.0, 2.0, P, dtype=np.float32)
    scores = np.arange(L * 8 * P, dtype=np.float32).reshape(L, 8, P)
    out = split_pair_scores(sa, an, idx, d, scores)
    assert len(out) == 3 and all(isinstance(o, LocalAttentionScores) for o in out)
    assert np.array_equal(out[0].site_offsets, [0, 3, 5]) and out[0].site_offsets.dtype == np.int32
    assert np.array_equal(out[1].site_offsets, [0, 0]) and out[1].neighbors.shape == (0,)
    assert out[1].scores.shape == (L, 8, 0)
    assert np.array_equal(out[2].site_offsets, [0, 2, 3, 5])
    assert np.array_equal(out[2].neighbors, idx[5:10]) and out[2].neighbors.dtype == np.int32
    assert np.array_equal(out[2].distances, d[5:10]) and out[2].distances.dtype == np.float32
    assert np.array_equal(out[2].scores, scores[:, :, 5:10])
    assert np.array_equal(np.concatenate([o.scores for o in out], axis=2), scores)
    with pytest.raises(ValueError, match="10 pairs"):
        split_pair_scores(sa, an, idx, d, scores[:, :, :9])
    with pytest.raises(ValueError, match="one CSR batch"):
        split_pair_scores(sa, an[:-1], idx, d, scores)


def test_local_attention_argument_is_checked_before_any_work():
    from scann_b200.engine import score_layout
    from scann_b200.model import ScannKerasModel
    assert score_layout(False) is None and score_layout(np.bool_(False)) is None
    assert score_layout(True) == "padded" and score_layout("padded") == "padded" and score_layout("csr") == "csr"
    with pytest.raises(ValueError, match="'padded' or 'csr'"):
        score_layout("dense")
    with pytest.raises(TypeError):
        score_layout(1)
    m = ScannKerasModel.__new__(ScannKerasModel)           # no engine: the check comes first
    with pytest.raises(TypeError, match="local_attention must be a bool"):
        m.predict({}, local_attention="yes")
    with pytest.raises(TypeError, match="local_attention must be a bool"):
        m.predict_structures([], local_attention=None)


def test_unpack_entry_points_refuse_bad_sizes():
    import ctypes
    from scann_b200 import _abi
    lib = _abi.lib
    buf = (ctypes.c_float * 64)()
    a = ctypes.addressof(buf)
    fake = 256                                              # never dereferenced: every call below is refused first
    cases = [
        (lambda: lib.scann_attn_to_padded(a, 0, 32, fake, fake, fake, 1, 1, 1, fake, None), "bad layer count"),
        (lambda: lib.scann_attn_to_padded(a, 1, 0, fake, fake, fake, 1, 1, 1, fake, None), "bad plan row count"),
        (lambda: lib.scann_attn_to_padded(a + 4, 1, 32, fake, fake, fake, 1, 1, 1, fake, None), "16-byte aligned"),
        (lambda: lib.scann_attn_to_padded(a, 1, 32, fake, fake, fake, 0, 1, 1, fake, None), "bad shape"),
        (lambda: lib.scann_attn_to_padded(a, 1, 32, fake, fake, fake, 1024, 1024, 512, fake, None), "exceed int32"),
        (lambda: lib.scann_attn_to_padded(a, 1, 32, None, fake, fake, 1, 1, 1, fake, None), "NULL"),
        (lambda: lib.scann_attn_to_padded(a, 1, 32, fake, fake, fake, 1, 1, 1, None, None), "NULL"),
        (lambda: lib.scann_attn_to_csr(a, 1, 32, fake, fake, 0, fake, None), "bad ld"),
        (lambda: lib.scann_attn_to_csr(a, 1, 32, None, fake, 32, fake, None), "NULL"),
        (lambda: lib.scann_attn_to_csr(None, 1, 32, fake, fake, 32, fake, None), "NULL"),
    ]
    for call, msg in cases:
        assert call() == 1
        assert msg in _abi.last_error(), (msg, _abi.last_error())


# ------------------------------------------------------------------------------------------------ GPU helpers
def _spec_model(cfg_name, L, seed=3, feature=None, **over):
    from scann_b200.config import model_spec
    from scann_b200.configs import get_config
    from scann_b200.model import create_model
    from scann_b200.params import ParamLayout
    cfg = get_config(cfg_name, feature=feature) if feature else get_config(cfg_name)
    cfg["model"]["n_attention"] = L
    cfg["model"].update(over)
    spec = model_spec(cfg)
    lay = ParamLayout(spec)
    arena = lay.randomize_arena(seed)
    return create_model(cfg, infer=True, arena=arena), spec, lay.to_dict(arena)


def oracle_attn(w, inputs, spec, dtype):
    """The oracle's per-layer local-attention scores, [L, B, 8, M, N] numpy."""
    import torch
    from oracle import scann_oracle as O
    from tests.golden.make_golden import oracle_kwargs
    kw = dict(oracle_kwargs(spec), use_ring=bool(spec.use_ring))
    with torch.no_grad():
        tw = {k: torch.tensor(np.asarray(v), dtype=dtype) for k, v in w.items()}
        _, _, trace = O.forward(tw, O.to_torch_inputs(inputs, dtype), return_all=True, **kw)
    return np.stack([trace[f"attn{l}"].numpy() for l in range(spec.n_attention)])


def check_against_oracle(la, inputs, spec, w, full_depth=False):
    """Valid rows within the ga_score bounds of test_gpu_parity against the fp64 oracle, masked slots exactly 0, rows
    without a valid slot exactly 1/N (as the fp32 oracle computes them: in fp64 the logits survive the -1e9), every
    row sums to 1."""
    import torch
    from tests.test_gpu_parity import TOL_OUT, rel
    L = spec.n_attention
    mask = np.asarray(inputs["neighbor_mask"]).astype(bool)
    B, M, N = mask.shape
    assert la.shape == (L, B, 8, M, N) and la.dtype == np.float32
    rows = la.transpose(0, 1, 3, 2, 4)                        # [L, B, M, 8, N]
    valid = mask.any(-1)                                     # [B, M]
    a64 = oracle_attn(w, inputs, spec, torch.float64).transpose(0, 1, 3, 2, 4)
    a32 = oracle_attn(w, inputs, spec, torch.float32).transpose(0, 1, 3, 2, 4)
    err = rel(rows[:, valid], a64[:, valid])
    tol = max(TOL_OUT, 5.0 * rel(a32[:, valid], a64[:, valid])) if full_depth else TOL_OUT
    assert err <= tol, (err, tol)
    masked = np.broadcast_to(~mask[:, :, None, :], rows.shape[1:])     # [B, M, 8, N]
    assert (rows[:, masked & valid[:, :, None, None]] == 0).all()
    assert (rows[:, ~valid] == np.float32(1.0) / np.float32(N)).all()
    assert np.allclose(a32[:, ~valid], 1.0 / N, rtol=1e-6)
    atoms = np.asarray(inputs["atom_mask"]).reshape(B, M).astype(bool)
    sums = rows[:, atoms].sum(-1, dtype=np.float64)
    assert np.abs(sums - 1.0).max() <= 1e-6
    return err


def to_csr(inputs, marker=None):
    """A padded batch as the CSR dict of ``DataIterator.csr_item``; ``marker = (b, m, n)`` inserts the padding marker
    1000 at slot n of atom (b, m)'s list (the list grows by one, the later entries keep their slots after it)."""
    atomic = np.asarray(inputs["atomic"])
    mask = np.asarray(inputs["neighbor_mask"]).astype(bool)
    B, M, N = mask.shape
    n_at = (atomic != 0).sum(1)
    sa, an, z, idx, wt, d = [0], [0], [], [], [], []
    for b in range(B):
        for m in range(int(n_at[b])):
            k = int(mask[b, m].sum())
            li = list(inputs["neighbors"][b, m, :k])
            lw = list(inputs["neighbor_weight"][b, m, :k])
            ld = list(inputs["neighbor_distance"][b, m, :k])
            if marker is not None and marker[:2] == (b, m):
                n = marker[2]
                li.insert(n, 1000)
                lw.insert(n, 1.0)
                ld.insert(n, 2.0)
            z.append(atomic[b, m])
            idx += li
            wt += lw
            d += ld
            an.append(len(idx))
        sa.append(len(z))
    an_a = np.asarray(an, np.int32)
    return {"struct_atom_off": np.asarray(sa, np.int32), "atom_nbr_off": an_a, "z": np.asarray(z, np.int32),
            "nbr_idx": np.asarray(idx, np.int32), "nbr_w": np.asarray(wt, np.float32),
            "nbr_d": np.asarray(d, np.float32), "M": int(n_at.max()), "N": int(np.diff(an_a).max())}


def wide_batch(B=6, seed=4):
    """QM9-like atoms with 33..48 neighbours each: the round-1 plan (N > 32)."""
    from scann_b200.synth import Shape, make_batch
    shape = Shape("wide", B, 20, 48, (8, 20), (1, 6, 7, 8, 9), None, (33, 48), (0.9, 4.0), (0.4, 3.0))
    inputs, _ = make_batch(shape, seed)
    inputs["neighbor_mask"][0, 3] = False                   # an atom without valid neighbours
    inputs["neighbors"][0, 3] = 0
    return inputs


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_the_flag_changes_neither_the_predictions_nor_the_default_graph():
    from scann_b200.synth import make_batch
    model, spec, _ = _spec_model("qm9", 3)
    inputs, _ = make_batch("qm9", 5, B=32)
    y0, ga0 = model.predict(inputs)
    eng = model.engine
    (b,) = eng._batches.values()
    n0 = b.graphs[("infer", True)].n_launches
    y1, ga1, la = model.predict(inputs, local_attention=True)
    assert np.array_equal(y0, y1) and np.array_equal(ga0, ga1)
    assert la.shape == (3, 32, 8, 29, 16)
    assert b.graphs[("infer", True)].n_launches == n0
    assert b.graphs[("infer", True, "padded")].n_launches == n0 + 1
    y2, ga2 = model.predict(inputs)
    assert np.array_equal(y0, y2) and np.array_equal(ga0, ga2)
    model.infer = False                                     # [y, la] outside infer mode
    y3, la3 = model.predict(inputs, local_attention=True)
    assert np.array_equal(y3, y0) and np.array_equal(la3, la)
    assert isinstance(model.predict(inputs), np.ndarray)
    model.infer = True
    structs = qm9_like(20, seed=3)
    ys, gas = model.predict_structures(structs, batch_size=8)
    ys1, gas1, las = model.predict_structures(structs, batch_size=8, local_attention=True)
    assert np.array_equal(ys, ys1) and all(np.array_equal(a, c) for a, c in zip(gas, gas1)) and len(las) == 20
    eng.check_status()


@pytest.mark.gpu
def test_qm9_l3_on_the_pipelined_plan_against_the_oracle():
    from scann_b200.synth import make_batch
    model, spec, w = _spec_model("qm9", 3)
    inputs, _ = make_batch("qm9", 6, B=16)
    inputs["neighbor_mask"][1, 2] = False                   # an atom without valid neighbours
    inputs["neighbors"][1, 2] = 0
    _, _, la = model.predict(inputs, local_attention=True)
    assert all(b.stride == 32 for b in model.engine._batches.values())
    check_against_oracle(la, inputs, spec, w)


@pytest.mark.gpu
def test_more_than_32_neighbours_on_the_round_1_plan_against_the_oracle():
    model, spec, w = _spec_model("qm9", 2)
    inputs = wide_batch()
    _, _, la = model.predict(inputs, local_attention=True)
    assert all(b.stride != 32 for b in model.engine._batches.values())
    check_against_oracle(la, inputs, spec, w)


@pytest.mark.gpu
@pytest.mark.parametrize("noup_pipe", ["1", "0"])
def test_no_geometry_update_with_ring_features_against_the_oracle(monkeypatch, noup_pipe):
    """model_ptgp.yaml family (g_update=False, use_ring) on the pipelined attention kernel and on the round-1 one."""
    from scann_b200.synth import make_batch
    monkeypatch.setenv("SCANN_NOUP_PIPE", noup_pipe)
    model, spec, w = _spec_model("ptgp", 3, seed=12, g_update=False, gaussian_d=4.0)
    assert spec.use_ring and not spec.g_update
    inputs, _ = make_batch("ptgp", 4, B=2, use_ring=True)
    _, _, la = model.predict(inputs, local_attention=True)
    check_against_oracle(la, inputs, spec, w)


@pytest.mark.gpu
def test_cgcnn_model_against_the_oracle():
    from scann_b200.synth import make_batch
    model, spec, w = _spec_model("qm9", 2, seed=13, feature="cgcnn")
    assert spec.feature == "cgcnn"
    inputs, _ = make_batch("qm9", 8, B=5, feature="cgcnn")
    _, _, la = model.predict(inputs, local_attention=True)
    check_against_oracle(la, inputs, spec, w)


@pytest.mark.gpu
def test_a_padding_marker_keeps_its_slot():
    from scann_b200.datagenerator import pack_padded
    from scann_b200.synth import make_batch
    model, spec, w = _spec_model("qm9", 2)
    base, _ = make_batch("qm9", 9, B=6)
    k = int(base["neighbor_mask"][2, 1].sum())
    csr = to_csr(base, marker=(2, 1, k // 2))
    inputs = pack_padded(csr)
    assert not inputs["neighbor_mask"][2, 1, k // 2] and inputs["neighbor_mask"][2, 1, k // 2 + 1]
    _, _, la = model.predict(csr, local_attention=True)
    check_against_oracle(la, inputs, spec, w)
    assert (la[:, 2, :, 1, k // 2] == 0).all() and (la[:, 2, :, 1, k // 2 + 1] > 0).all()
    _, _, la_pad = model.predict(inputs, local_attention=True)          # the padded dict of the same batch
    assert np.array_equal(la, la_pad)


@pytest.mark.gpu
def test_full_depth_qm9_batch_against_the_oracle():
    from scann_b200.synth import make_batch
    model, spec, w = _spec_model("qm9", 7, seed=21)
    inputs, _ = make_batch("qm9", 13, B=128)
    _, _, la = model.predict(inputs, local_attention=True)
    check_against_oracle(la, inputs, spec, w, full_depth=True)


def host_scores(model, structs, batch_size):
    """predict(csr, local_attention=True) on the host-built batches with predict_structures' shape classes, read at
    the valid slots in list order: [L, 8, P] per structure, and the host CSR lists."""
    from scann_b200.model import shape_class
    it = host_iterator(structs, 4.0, 0.4, bool(model.spec.g_update), batch_size)
    out = []
    for i in range(len(it)):
        csr, _ = it.csr_item(i)
        csr = dict(csr)
        csr["M"], csr["N"] = shape_class(csr["M"], csr["N"])
        _, _, la = model.predict(csr, local_attention=True)
        sa, an = csr["struct_atom_off"], csr["atom_nbr_off"]
        for s in range(len(sa) - 1):
            cols = [la[:, s, :, m, :an[sa[s] + m + 1] - an[sa[s] + m]] for m in range(sa[s + 1] - sa[s])]
            out.append((np.concatenate(cols, axis=2), an[sa[s]:sa[s + 1] + 1] - an[sa[s]],
                        csr["nbr_idx"][an[sa[s]]:an[sa[s + 1]]], csr["nbr_d"][an[sa[s]]:an[sa[s + 1]]]))
    return out


@pytest.mark.gpu
def test_structures_route_equals_the_host_route():
    from scann_b200 import voronoi as V
    from tests.test_gpu_parity import TOL_OUT, rel
    model, _ = _model("qm9")
    spec = model.spec
    structs = qm9_like(40, seed=11)
    structs[17:17] = [hub()]                               # a batch with > 32 neighbours: the 64-row plan
    structs.append(lone_atom())                            # a site without kept neighbours (y is NaN)
    y, ga, la = model.predict_structures(structs, batch_size=16, local_attention=True)
    want = host_scores(model, structs, 16)
    lists = V.compute_voronoi_neighbors(structs)
    assert len(la) == len(structs) == len(want)
    for k, (got, (sc, off, nb, d), lst) in enumerate(zip(la, want, lists)):
        assert np.array_equal(got.scores, sc), k
        assert np.array_equal(got.site_offsets, off) and np.array_equal(got.neighbors, nb), k
        assert np.array_equal(got.distances.view(np.uint32), d.view(np.uint32)), k
        assert got.scores.shape == (spec.n_attention, 8, sum(len(x) for x in lst))
        assert np.array_equal(np.diff(got.site_offsets), [len(x) for x in lst]), k
        assert np.array_equal(got.neighbors, [t[1] for x in lst for t in x]), k
        assert np.array_equal(got.distances, np.float32([t[4] for x in lst for t in x])), k
    assert la[-1].scores.shape == (spec.n_attention, 8, 0)
    eng = model.engine
    assert any(b.N > 32 for b in eng._batches.values())
    for g in la:                                           # the softmax of every site with neighbours sums to 1
        off = g.site_offsets
        c = np.concatenate([np.zeros(g.scores.shape[:2] + (1,)), np.cumsum(g.scores, axis=2, dtype=np.float64)], 2)
        sums = (c[..., off[1:]] - c[..., off[:-1]])[..., np.diff(off) > 0]
        assert sums.size == 0 or np.abs(sums - 1.0).max() <= 1e-6
    for bs in (1, 7, 128):
        y2, ga2, la2 = model.predict_structures(structs, batch_size=bs, local_attention=True)
        assert np.array_equal(y2, model.predict_structures(structs, batch_size=bs)[0], equal_nan=True)
        assert rel(np.concatenate([g.scores for g in la2], axis=2),
                   np.concatenate([g.scores for g in la], axis=2)) <= TOL_OUT
        assert all(np.array_equal(a.neighbors, c.neighbors) for a, c in zip(la2, la))
    from scann.models import SCANN
    facade = SCANN.__new__(SCANN)
    facade.model, facade.mean, facade.std = model, 2.5, 4.0
    y3, ga3, la3 = facade.predict_structures(structs, batch_size=16, local_attention=True)
    assert np.array_equal(y3, y * np.float32(4.0) + 2.5, equal_nan=True) and all(np.array_equal(a.scores, c.scores)
                                                                 for a, c in zip(la3, la))


@pytest.mark.gpu
def test_graph_replay_equals_eager():
    from scann_b200.synth import make_batch
    model, _, _ = _spec_model("qm9", 3)
    inputs, _ = make_batch("qm9", 2, B=24)
    structs = qm9_like(30, seed=4)
    first = model.predict(inputs, local_attention=True)          # capture
    replay = model.predict(inputs, local_attention=True)
    s_first = model.predict_structures(structs, batch_size=16, local_attention=True)
    s_replay = model.predict_structures(structs, batch_size=16, local_attention=True)
    model.engine.use_graphs = False
    eager = model.predict(inputs, local_attention=True)
    s_eager = model.predict_structures(structs, batch_size=16, local_attention=True)
    for a, b, c in zip(first, replay, eager):
        assert np.array_equal(a, b) and np.array_equal(a, c)
    for run in (s_replay, s_eager):
        assert np.array_equal(run[0], s_first[0])
        assert all(np.array_equal(a.scores, c.scores) for a, c in zip(run[2], s_first[2]))


@pytest.mark.gpu
def test_a_thousand_molecules_with_scores_stay_within_the_shape_class_cache():
    model, _ = _model("qm9")
    eng = model.engine
    structs = qm9_like(1000, seed=21)
    y, ga, la = model.predict_structures(structs, batch_size=128, local_attention=True)
    assert len(la) == 1000 and np.isfinite(y).all()
    assert eng.shape_class_evictions == 0
    assert eng.graph_captures == len(eng._batches) <= eng.max_shape_classes, sorted(eng._batches)
    y2, _ = model.predict_structures(structs, batch_size=128)       # the graphs without scores: separate captures
    assert np.array_equal(y, y2)
    assert eng.graph_captures == 2 * len(eng._batches) and eng.shape_class_evictions == 0
    n0 = eng.graph_captures
    model.predict_structures(structs, batch_size=128, local_attention=True)
    model.predict_structures(structs, batch_size=128)
    assert eng.graph_captures == n0 and eng.shape_class_evictions == 0
