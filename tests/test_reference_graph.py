"""The reference's OWN floating-point graph code, run here, against the oracle, the committed goldens and the
parameter layout (SURVEY.md 8c; VERDICT round 1 "what's weak" 1: "the floating-point rows stay unpinned").

TensorFlow is not installable in this image, so ``tests/tf_shim.py`` supplies the TensorFlow / Keras PRIMITIVES
(Dense, LayerNormalization, softmax, einsum, gather_nd ...: restated from their documented semantics on PyTorch-CPU)
and the reference's modules are imported from the checkout named by SCANN_REFERENCE_ROOT on top of it, UNMODIFIED:

  * ``create_model(config)``                     scann/models/scann_model.py:329-453
  * ``LocalAttention / GlobalAttention / ResidualNorm .call``   scann/layers/attention.py:19-318
  * ``GaussianExpansion.call``, ``gather_shape``, ``mrelu``      scann/layers/custom_layers.py:6-65
  * ``root_mean_squared_error``                  scann/layers/losses.py:5-6

Every expression the reference wrote -- layer order, einsum strings, reshapes, mask arithmetic, concat order,
residuals, which kernels carry ``l2(1e-4)``, where the three Dropout sites sit, where ``ga_score`` comes from --
therefore executes as written, forward and backward (torch autograd), and is compared with
``oracle/scann_oracle.py`` at fp64 round-off, with ``tests/golden/*.npz`` (the expected values of the GPU tests) and
with ``scann_b200/params.py`` (weight inventory, shapes, l2 flags).  Parity status after this file: graph wiring
pinned to reference-run code; primitive kernels of TensorFlow itself (its fp32 summation order) remain unpinned.

The values these comparisons found are stored in ``tests/golden/reference/graph_*.npz`` (recorded from this repo's
oracle and layout as last compared equal with the reference); without the checkout the tests check against them,
and the few that need the reference's own code to run skip.
"""
import os
import warnings

import numpy as np
import pytest
import torch

from oracle import scann_oracle as O
from scann_b200.config import model_spec
from scann_b200.configs import get_config
from scann_b200.params import ParamLayout
from scann_b200.synth import make_batch
from tests.golden.make_golden import CASES, build_case, oracle_kwargs
from tests.golden.make_reference_golden import pack
from tests.ref_stubs import SKIP_REASON, check_stored, load_reference_graph, reference_available

needs_reference = pytest.mark.skipif(not reference_available(), reason=SKIP_REASON)
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def ref():
    """The reference's own graph code, or None where its source is absent (the stored values stand in)."""
    if not reference_available():
        return None
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")          # the reference's own SyntaxWarnings (regex escapes)
        return load_reference_graph()


def run_reference_graph(ref, cfg, w_np, inputs, target, dtype=torch.float64, drop_masks=None, grads=True):
    """create_model(cfg) of the reference on the shim -> dict(y, ga, loss, grads, session)."""
    shim = ref["shim"]
    wt = {k: torch.tensor(np.asarray(v, np.float64), dtype=dtype, requires_grad=grads) for k, v in w_np.items()}
    with shim.session(inputs, wt, dtype=dtype, drop_masks=drop_masks) as s:
        model = ref["create_model"](cfg)
        y = model.outputs[0]                                                   # [B,1]
        ga = model.get_layer("global_attention").output[0]                     # scann_model.py:82 -> [B,M,1]
        out = {"y": y.detach().numpy(), "ga": ga.detach().numpy(), "session": s, "weights": wt}
        if grads:
            t = torch.tensor(np.asarray(target, np.float64), dtype=dtype).reshape(-1, 1)
            loss = ref["root_mean_squared_error"](t, y) + sum(model.losses)    # Keras adds the regulariser penalties
            loss.backward()
            out["loss"] = float(loss.detach())
            out["grads"] = {k: (v.grad.numpy() if v.grad is not None else np.zeros(v.shape)) for k, v in wt.items()}
    return out


def oracle_run(spec, lay, w, inputs, target, **extra):
    l2n = [e.name for e in lay if e.l2]
    kw = dict(oracle_kwargs(spec), use_ring=spec.use_ring, mrelu_head=spec.mrelu_head)
    kw.update(extra)
    return O.loss_and_grads(w, inputs, target, l2n, dtype=torch.float64, **kw)


def compact(lay, w, inputs, target, y, ga, loss, grads):
    """What a graph comparison stores: ``make_reference_golden.pack`` (outputs, loss, per-tensor max|grad| and
    ||grad||_2) with the flat gradient arena sampled at every 1040th element instead of every 13th, to keep it small."""
    z = pack(lay, lay.from_dict(w), inputs, target, y, ga, loss, grads)
    z["grad_idx"], z["grad_sample"] = z["grad_idx"][::80], z["grad_sample"][::80]
    return z


def relerr(a, r):
    a, r = np.asarray(a, np.float64), np.asarray(r, np.float64)
    return float(np.abs(a - r).max() / max(np.abs(r).max(), 1e-300))


def case(cfg_name, shape, B, L, pseed, bseed, *, target="homo", feature="atomic", use_drop=False, **model_over):
    cfg = get_config(cfg_name, target=target, feature=feature, use_drop=use_drop)
    cfg["model"].update(model_over)
    if L is not None:
        cfg["model"]["n_attention"] = L
    spec = model_spec(cfg)
    lay = ParamLayout(spec)
    w = lay.to_dict(lay.randomize_arena(pseed))
    inputs, tgt = make_batch(shape, bseed, B=B, use_ring=spec.use_ring, feature=feature)
    return cfg, spec, lay, w, inputs, tgt


GRAPH_CASES = {
    # SCANN+ (g_update=True) on the three shipped shapes
    "qm9_l2": dict(cfg_name="qm9", shape="qm9", B=5, L=2, pseed=2, bseed=10),
    "mp2018_l3": dict(cfg_name="mp2018", shape="mp2018", B=3, L=3, pseed=3, bseed=11),
    "fullerene_no_ga_norm": dict(cfg_name="fullerene", shape="fullerene", B=2, L=2, pseed=4, bseed=12),
    # SCANN (g_update=False) with ring features: attention.py:155, scann_model.py:367-371,391
    "ptgp_noupdate_ring": dict(cfg_name="ptgp", shape="qm9", B=4, L=3, pseed=5, bseed=13, g_update=False, gaussian_d=4.0),
    # feature == 'cgcnn' (scann_model.py:364-365), target e_b -> mrelu head (scann_model.py:446, custom_layers.py:6-15)
    "qm9_cgcnn": dict(cfg_name="qm9", shape="qm9", B=3, L=2, pseed=6, bseed=14, feature="cgcnn"),
    "qm9_mrelu_head": dict(cfg_name="qm9", shape="qm9", B=6, L=2, pseed=7, bseed=15, target="e_b"),
    # no ResidualNorm between the attention layers (scann_model.py:404-408)
    "qm9_no_attn_norm": dict(cfg_name="qm9", shape="qm9", B=3, L=2, pseed=8, bseed=16, use_attn_norm=False),
}


@pytest.mark.parametrize("name", list(GRAPH_CASES))
def test_reference_create_model_matches_oracle(ref, name):
    """Forward, ga_score, loss and EVERY per-tensor gradient of the reference's own graph = the oracle's (fp64)."""
    cfg, spec, lay, w, inputs, target = case(**GRAPH_CASES[name])
    loss, y, ga, grads = oracle_run(spec, lay, w, inputs, target)
    check_stored(f"graph_{name}", compact(lay, w, inputs, target, y, ga, loss, grads), rtol=1e-10, atol=1e-15)
    if spec.mrelu_head:
        assert (y >= 0).all() and (y == 0).any(), "case must exercise the clipped branch of mrelu"
    if ref is None:
        return
    r = run_reference_graph(ref, cfg, w, inputs, target)
    assert r["y"].shape == y.shape and r["ga"].shape == ga.shape
    np.testing.assert_allclose(r["y"], y, rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(r["ga"], ga, rtol=1e-11, atol=1e-15)
    assert abs(r["loss"] - loss) <= 1e-12 * max(1.0, abs(loss))
    assert set(grads) == set(r["grads"])
    for k in grads:
        assert relerr(r["grads"][k], grads[k]) <= 1e-10 or np.abs(grads[k]).max() < 1e-14, k


@pytest.mark.parametrize("name", ["qm9_l2", "ptgp_noupdate_ring", "qm9_cgcnn", "qm9_no_attn_norm"])
def test_reference_weight_inventory_matches_param_layout(ref, name):
    """The reference graph asks for exactly the tensors of scann_b200/params.py (names, shapes: checked by the
    shim at every request), declares exactly the fed inputs, and puts l2(1e-4) on exactly the layout's l2 kernels."""
    cfg, spec, lay, w, inputs, target = case(**GRAPH_CASES[name])
    sites = ["dropout"] + [f"{O._name('residual_norm', l)}/dropout" for l in range(spec.n_attention) if spec.use_attn_norm]
    mine = {"weights": sorted(e.name for e in lay), "shapes": np.array([e.size for e in sorted(lay, key=lambda e: e.name)]),
            "l2": sorted(e.name for e in lay if e.l2), "inputs": sorted(inputs), "dropout_sites": sorted(sites)}
    check_stored(f"graph_inventory_{name}", mine)
    if ref is None:
        return
    r = run_reference_graph(ref, cfg, w, inputs, target, grads=False)
    s = r["session"]
    assert sorted(s.used_weights) == mine["weights"]
    assert sorted(n for n, _ in s.reg_losses) == mine["l2"]
    assert sorted(s.inputs_asked) == mine["inputs"]
    assert sorted(s.dropout_sites) == mine["dropout_sites"]      # use_drop=False: no attention-probability Dropout


@needs_reference
@pytest.mark.parametrize("name", list(CASES))
def test_golden_vectors_equal_the_reference_graph(ref, name):
    """tests/golden/*.npz -- the expected values of the GPU parity tests -- against the reference's own graph run on
    the same seeded case: the fixtures are pinned to reference-run code, not only to the restatement."""
    cfg, spec, lay, arena, inputs, target = build_case(name)
    z = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    r = run_reference_graph(ref, cfg, lay.to_dict(arena), inputs, target)
    np.testing.assert_allclose(r["y"], z["y"], rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(r["ga"], z["ga"], rtol=1e-10, atol=1e-14)
    assert abs(r["loss"] - float(z["loss"])) < 1e-10
    garena = lay.from_dict({k: v.astype(np.float32) for k, v in r["grads"].items()})
    np.testing.assert_allclose(garena[z["grad_idx"]], z["grad_sample"], rtol=1e-6, atol=1e-9)
    l2 = np.sqrt(sum((g.astype(np.float64) ** 2).sum() for g in r["grads"].values()))
    assert abs(l2 - float(z["grad_l2norm"])) <= 1e-9 * float(z["grad_l2norm"])


def test_reference_dropout_sites_with_injected_masks(ref):
    """Training mode (use_drop=True): the three Dropout sites of the reference -- Dropout(0.1) behind dense_embed
    (scann_model.py:374), Dropout(0.1) inside every ResidualNorm (attention.py:29), Dropout(0.05) on the attention
    probabilities (attention.py:113,190-191) -- with the SAME masks injected into the reference graph and the oracle."""
    cfg, spec, lay, w, inputs, target = case("qm9", "qm9", 4, 2, 9, 17, use_drop=True)
    B, M, N = inputs["neighbors"].shape
    rng = np.random.default_rng(5)

    def mask(shape, rate):
        return (rng.random(shape) >= rate).astype(np.float64) / (1.0 - rate)

    dm_oracle, dm_ref = {"dense_embed": mask((B, M, 128), 0.1)}, {}
    dm_ref["dropout"] = dm_oracle["dense_embed"]
    for l in range(spec.n_attention):
        rn, la = O._name("residual_norm", l), O._name("local_attention", l)
        dm_oracle[rn] = dm_ref[f"{rn}/dropout"] = mask((B, M, 128), 0.1)
        dm_oracle[la] = dm_ref[f"{la}/drop_out"] = mask((B, 8, M, N), 0.05)
    loss, y, ga, grads = oracle_run(spec, lay, w, inputs, target,
                                    drop_masks={k: torch.tensor(v) for k, v in dm_oracle.items()})
    y0 = oracle_run(spec, lay, w, inputs, target)[1]
    assert np.abs(y0 - y).max() > 1e-3, "the masks must matter"
    check_stored("graph_dropout_masks", dict(compact(lay, w, inputs, target, y, ga, loss, grads),
                                             sites=np.array(sorted(dm_ref))), rtol=1e-10, atol=1e-15)
    if ref is None:
        return
    r = run_reference_graph(ref, cfg, w, inputs, target, drop_masks={k: torch.tensor(v) for k, v in dm_ref.items()})
    assert sorted(r["session"].dropout_sites) == sorted(dm_ref)
    np.testing.assert_allclose(r["y"], y, rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(r["ga"], ga, rtol=1e-11, atol=1e-15)
    assert abs(r["loss"] - loss) <= 1e-12
    for k in grads:
        assert relerr(r["grads"][k], grads[k]) <= 1e-10, k


def test_reference_ptgp_yaml_as_shipped_raises_keyerror(ref):
    """configs/model_ptgp.yaml ships without g_update / gaussian_d: the reference's create_model raises KeyError
    (scann_model.py:378-380); scann_b200.config.model_spec keeps that behaviour."""
    cfg = get_config("ptgp")
    with pytest.raises(KeyError):
        model_spec(cfg)
    if ref is None:
        return
    inputs, _ = make_batch("qm9", 1, B=2, use_ring=True)
    with ref["shim"].session(inputs, {}):
        with pytest.raises(KeyError):
            ref["create_model"](cfg)


def test_reference_layers_edge_cases_match_oracle(ref):
    """Layer level, the edge cases the kernels special-case: an atom without a single valid neighbour
    (context = q, attention.py:206-214), fully padded atoms, a single-atom structure (tf.linalg.normalize gives 0/0 =
    NaN in ga_score and the prediction, attention.py:300-303) -- reference layers vs oracle functions."""
    rng = np.random.default_rng(3)
    B, M, N, D = 3, 6, 5, 128
    x = rng.standard_normal((B, M, D))
    g = rng.standard_normal((B, M, N, D))
    nbr = rng.integers(0, M, size=(B, M, N))
    nmask = rng.random((B, M, N)) < 0.7
    nmask[0, 1] = False                       # atom without neighbours
    nmask[1, 4:] = False                      # padded atoms
    amask = np.ones((B, M, 1), bool)
    amask[1, 4:] = False
    amask[2, 1:] = False                      # single-atom structure
    spec = model_spec(get_config("qm9"))
    lay = ParamLayout(spec)
    w = lay.to_dict(lay.randomize_arena(11))
    wt = {k: torch.tensor(v, dtype=torch.float64) for k, v in w.items()}
    xt, gt = torch.tensor(x), torch.tensor(g)
    o_idx = O.gather_shape(torch.tensor(nbr))
    o_attn, o_ctx, o_g = O.local_attention(wt, "local_attention", xt, o_idx, gt, torch.tensor(nmask, dtype=torch.float64),
                                           None, g_update=True)
    o_rn = O.residual_norm(wt, "residual_norm", o_ctx)
    o_ga, o_rep = O.global_attention(wt, "global_attention", o_rn, torch.tensor(amask, dtype=torch.float64), norm=True)
    o_rbf = O.gaussian_expansion(torch.tensor(np.abs(x[..., :N])), O.rbf_centers(4.0))
    assert np.isnan(o_ga.numpy()[2]).all() and not np.isnan(o_ga.numpy()[:2]).any()
    check_stored("graph_layer_edge_cases", {"idx": o_idx.numpy(), "attn": o_attn.numpy(), "ctx": o_ctx.numpy()[..., ::8],
                                            "g": o_g.numpy()[..., ::8], "rn": o_rn.numpy()[..., ::8], "rbf": o_rbf.numpy(),
                                            "ga": o_ga.numpy(), "rep": o_rep.numpy()[:2]}, rtol=1e-12, atol=1e-14)
    if ref is None:
        return
    shim = ref["shim"]
    with shim.session({}, wt) as s:
        la = ref["LocalAttention"](v_proj=False, kq_proj=True, dim=D, num_head=8, activation="swish", dropout=False,
                                   g_update=True)
        idx = ref["gather_shape"](torch.tensor(nbr))
        attn, ctx, g_new = la(xt, idx, gt, torch.tensor(nmask, dtype=torch.float64))
        rn = ref["ResidualNorm"](D)(ctx)
        ga_layer = ref["GlobalAttention"](v_proj=False, kq_proj=True, dim=D, norm=True)
        ga, rep = ga_layer(rn, torch.tensor(amask, dtype=torch.float64))
        rbf = ref["GaussianExpansion"](np.linspace(0, 4.0, 20, dtype="float32"))(torch.tensor(np.abs(x[..., :N])))
    assert torch.equal(idx, o_idx)
    for a, b in ((attn, o_attn), (ctx, o_ctx), (g_new, o_g), (rn, o_rn), (rbf, o_rbf)):
        np.testing.assert_allclose(a.numpy(), b.numpy(), rtol=1e-12, atol=1e-14)
    np.testing.assert_array_equal(np.isnan(ga.numpy()), np.isnan(o_ga.numpy()))
    np.testing.assert_allclose(ga.numpy()[:2], o_ga.numpy()[:2], rtol=1e-12, atol=1e-16)
    np.testing.assert_allclose(rep.numpy()[:2], o_rep.numpy()[:2], rtol=1e-12, atol=1e-14)


@needs_reference
def test_reference_graph_in_fp32_sets_the_noise_floor(ref):
    """The reference computes in fp32.  Its own graph run in fp32 on the shim sits as far from fp64 truth as the fp32
    oracle does -- the floor the GPU tests' full-depth tolerances are normalised by (DESIGN.md section 5)."""
    cfg, spec, lay, arena, inputs, target = build_case("qm9_b4")
    w = lay.to_dict(arena)
    r32 = run_reference_graph(ref, cfg, w, inputs, target, dtype=torch.float32, grads=False)
    y64, ga64 = O.predict(w, inputs, torch.float64, **oracle_kwargs(spec))
    y32, ga32 = O.predict(w, inputs, torch.float32, **oracle_kwargs(spec))
    e_ref, e_orc = relerr(r32["y"], y64), relerr(y32, y64)
    assert 1e-8 < e_ref <= 2e-5 and e_ref <= 3 * e_orc + 1e-6 and e_orc <= 3 * e_ref + 1e-6
    assert relerr(r32["ga"], ga64) <= 1e-5


def _graph_layers(ref, cfg, spec, lay, w, inputs):
    """Top-level layers of the reference's create_model run, in graph (call) order."""
    r = run_reference_graph(ref, cfg, w, inputs, None, grads=False)
    return list(r["session"].top_layers.items())


@pytest.mark.parametrize("name", ["qm9_l2", "ptgp_noupdate_ring", "qm9_cgcnn", "qm9_mrelu_head", "qm9_no_attn_norm"])
def test_arena_order_and_model_config_follow_the_reference_graph(ref, name):
    """(1) ``ParamLayout`` lists the tensors in the reference's Keras order: layers in graph order, inside a layer its
    own variables, then its sub-layers in attribute-assignment order (attention.py:25-35,95-113,260-262) -- the
    ``weight_names`` order of a Keras HDF5 file.  (2) The ``model_config`` JSON that ``model.save`` writes names the
    same layers (class, name) in the same order, and carries every key / value of the reference layers' OWN
    ``get_config()`` (attention.py:42-50,218-231,320-331; custom_layers.py:67-75)."""
    import json
    from scann_b200.model import keras_model_config, spec_from_model_config
    cfg, spec, lay, w, inputs, target = case(**GRAPH_CASES[name])
    mc = json.loads(keras_model_config(spec))["config"]["layers"]
    import dataclasses
    want = dataclasses.replace(spec, n_atoms=0) if spec.feature == "cgcnn" else spec     # cgcnn graphs have no vocabulary
    assert spec_from_model_config(json.dumps({"config": {"layers": mc}})) == want
    check_stored(f"graph_arena_order_{name}", {"order": np.array([e.name for e in lay]),
                                               "model_config": np.array(json.dumps(mc, sort_keys=True))})
    if ref is None:
        return
    with ref["shim"].session(inputs, {k: torch.tensor(v, dtype=torch.float64) for k, v in w.items()}) as s:
        ref["create_model"](cfg)
        layers = list(s.top_layers.items())
        order = [n for _, l in layers for n in l.weights_order()]
        ref_cfg = {n: (type(l).__name__, l.get_config()) for n, l in layers}
    assert order == [e.name for e in lay]
    skip = {"Lambda", "Multiply"}                              # wiring-only layers are not in the written config
    assert [(c, n) for n, (c, _) in ref_cfg.items() if c not in skip] == [(l["class_name"], l["name"]) for l in mc]
    for l in mc:
        cls, rc = ref_cfg[l["name"]]
        for k, v in rc.items():
            if k == "activation" and callable(v):
                v = v.__name__
            got = l["config"][k]
            if k == "centers":
                np.testing.assert_allclose(np.asarray(got), np.asarray(v, np.float64), rtol=1e-6)
            else:
                assert got == v, (l["name"], k, got, v)


def test_layer_mirrors_keep_the_reference_constructor_config_and_weight_order(ref):
    """scann_b200.layers.{LocalAttention, ResidualNorm, GlobalAttention, GaussianExpansion}: same constructor
    arguments, same ``get_config`` items and the same ``set_weights`` order as the reference's own classes."""
    import json
    from scann_b200 import layers as mine
    la_kw = dict(v_proj=False, kq_proj=True, dim=128, num_head=8, activation="swish", dropout=False, g_update=True)
    ga_kw = dict(v_proj=False, kq_proj=True, dim=128, norm=False)
    centers = np.linspace(0, 4.0, 20, dtype="float32")
    ours = [mine.LocalAttention(**la_kw), mine.ResidualNorm(128), mine.GlobalAttention(**ga_kw),
            mine.GaussianExpansion(centers)]
    assert ours[3].width == 0.25
    stored = {}
    for layer in ours:
        c = {k: np.asarray(v).tolist() for k, v in layer.get_config().items() if k != "name"}
        stored[type(layer).__name__] = np.array(json.dumps(c, sort_keys=True))
        stored[type(layer).__name__ + "/weights"] = np.array(list(getattr(layer, "weight_names", [])) or [""])
    check_stored("graph_layer_mirrors", stored)
    if ref is None:
        return
    shim = ref["shim"]
    spec = model_spec(get_config("qm9"))
    lay = ParamLayout(spec)
    wt = {k: torch.tensor(v, dtype=torch.float64) for k, v in lay.to_dict(lay.randomize_arena(1)).items()}
    with shim.session({}, wt):
        pairs = [(ref["LocalAttention"](**la_kw), ours[0]), (ref["ResidualNorm"](128), ours[1]),
                 (ref["GlobalAttention"](**ga_kw), ours[2]), (ref["GaussianExpansion"](centers), ours[3])]
        for theirs, ours_ in pairs:
            a = {k: v for k, v in theirs.get_config().items() if k != "name"}
            b = {k: v for k, v in ours_.get_config().items() if k != "name"}
            assert set(a) == set(b), type(theirs).__name__
            for k in a:
                assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), (type(theirs).__name__, k)
            if hasattr(ours_, "weight_names"):
                p = theirs.path()
                assert [n[len(p) + 1:] for n in theirs.weights_order()] == list(ours_.weight_names)
        assert pairs[3][0].width == 0.25


# ------------------------------------------------------------------------------------------------ training shell
class _FakeHistory:
    def __init__(self):
        self.history = {"loss": [0.9, 0.5, 0.4], "mae": [0.7, 0.31, 0.33], "val_mae": [0.8, 0.45, 0.41]}


class _FakeModel:
    """Stands in for the compiled Keras model / the accelerated model: records what the shell asks of it."""

    def __init__(self, log):
        self.log = log

    def compile(self, **kw):
        self.log["compile"] = kw

    def fit(self, x, **kw):
        self.log["fit"] = (x, kw)
        return _FakeHistory()

    def load_weights(self, path):
        self.log["loaded"] = path

    def predict(self, inputs):
        return (inputs["neighbor_distance"].sum((1, 2)) * 0.01 - inputs["atomic"].sum(1) * 0.003).reshape(-1, 1)


class _Iter:
    def __init__(self, n_batches, seed):
        self.b = [make_batch("qm9", seed + i, B=3) for i in range(n_batches)]

    def __len__(self):
        return len(self.b)

    def __getitem__(self, i):
        return self.b[i]


def _numbers(obj):
    return {k: v for k, v in vars(obj).items() if isinstance(v, (int, float, str, bool)) and not k.startswith("_")}


@pytest.mark.parametrize("scheduler", ["sgdr", "cosine"])
def test_training_shell_follows_the_reference_train_and_evaluate(ref, scheduler, tmp_path, monkeypatch):
    """The reference's own ``SCANN.create_callbacks`` / ``train`` / ``evaluate`` (scann_model.py:163-313) executed
    with recording stand-ins for Keras' compile / fit / callbacks / optimisers, beside ``scann_b200.model.SCANN``'s:
    same callbacks with the same arguments, same learning-rate schedule arguments, same ``config.yaml``, the best
    checkpoint reloaded from the same path before evaluation (the reference deletes its model after fit), same
    ``report.txt`` and ``hist_data.npy``.  Without the reference, this repo's side is checked against what the
    comparison found (tests/golden/reference/graph_training_shell_*.npz)."""
    import json
    import yaml
    from scann_b200 import callbacks as C
    from scann_b200 import model as mine
    epochs = 40

    def run(who):
        root = tmp_path / who
        root.mkdir()
        log = {}
        cfg = get_config("qm9")
        cfg["hyper"].update(save_path=str(root / "run"), scheduler=scheduler, lr=5e-4, min_lr=1e-4)
        obj = object.__new__(ref["SCANN"] if who == "reference" else mine.SCANN)
        obj.config, obj.mean, obj.std = cfg, 0.25, 1.5
        obj.model = _FakeModel(log)
        obj.trainIter, obj.validIter, obj.testIter = _Iter(5, 100), _Iter(2, 200), _Iter(3, 300)
        if who == "reference":
            with ref["shim"].session({}, {}):
                obj.train(epochs=epochs)
                assert not hasattr(obj, "model")                       # scann_model.py:243-245
                monkeypatch.setattr(ref["scann_model"], "load_model",
                                    lambda path, custom_objects=None: (log.__setitem__("loaded", path), _FakeModel(log))[1])
                obj.evaluate()
        else:
            obj.train(epochs=epochs)
            (root / "run_homo" / "models" / "model_homo.h5").write_bytes(b"")   # what ModelCheckpoint would have left
            obj.evaluate()
        d = dict(log=log, root=root, cfg=yaml.safe_load(open(root / "run_homo" / "config.yaml")),
                 report=open(root / "run_homo" / "report.txt").read(),
                 hist=np.load(root / "run_homo" / "hist_data.npy", allow_pickle=True))
        d["cfg"]["hyper"].pop("save_path")                             # config.yaml: compared up to the run directory
        return d

    m = run("mine")
    (xm, km), cm = m["log"]["fit"], m["log"]["fit"][1]["callbacks"]
    lr_mine = m["log"]["compile"]["optimizer"]
    # the values the comparison with the reference's shell checks, on every machine
    assert os.path.relpath(m["log"]["loaded"], m["root"]) == os.path.join("run_homo", "models", "model_homo.h5")
    assert (cm[0].monitor, cm[0].save_weights_only, cm[0].save_best_only) == ("val_mae", False, True)
    assert (cm[1].monitor, cm[1].patience) == ("val_mae", 200)
    assert len(xm) == 5 and km["epochs"] == epochs and len(km["validation_data"]) == 2
    if scheduler == "sgdr":
        assert lr_mine == 5e-4 and isinstance(cm[2], C.SGDRC) and cm[3].schedule.__self__ is cm[2]   # lr.lr_scheduler
    else:
        assert isinstance(lr_mine, mine.CosineDecay)
        assert (lr_mine.lr0, lr_mine.decay_steps, lr_mine.alpha) == (5e-4, 0.5 * 5 * epochs, 1e-4 / 5e-4)
    check_stored(f"graph_training_shell_{scheduler}", {
        "config": np.array(json.dumps(m["cfg"], sort_keys=True)), "report": np.array(m["report"]),
        "checkpoint": np.array(os.path.relpath(cm[0].filepath, m["root"])),
        "callbacks": np.array([type(c).__name__ for c in cm]),
        "sgdrc": np.array(json.dumps(_numbers(cm[2]) if scheduler == "sgdr" else {}, sort_keys=True)),
        "hist_true": np.asarray(m["hist"][1], np.float64), "hist_history": np.array(json.dumps(m["hist"][2], sort_keys=True))})
    check_stored(f"graph_training_shell_{scheduler}_pred", {"hist_pred": np.asarray(m["hist"][0], np.float64)}, rtol=1e-12)
    if ref is None:
        return
    r = run("reference")
    assert r["cfg"] == m["cfg"]
    # best checkpoint path relative to the run root
    assert os.path.relpath(r["log"]["loaded"], r["root"]) == os.path.relpath(m["log"]["loaded"], m["root"])
    # learning rate: a float under SGDR (the callback drives it), CosineDecay(lr, 0.5 * steps * epochs, alpha) otherwise
    adam = r["log"]["compile"]["optimizer"]
    assert type(adam).__name__ == "Adam" and adam.kwargs == {"decay": 1e-5}
    assert r["log"]["compile"]["loss"] is ref["scann_model"].root_mean_squared_error
    lr_ref = adam.args[0]
    if scheduler == "sgdr":
        assert lr_ref == lr_mine
    else:
        assert type(lr_ref).__name__ == "CosineDecay"
        assert lr_ref.args == (lr_mine.lr0, lr_mine.decay_steps) and lr_ref.kwargs["alpha"] == lr_mine.alpha
    # fit: same iterators, epochs, callbacks
    xr, kr = r["log"]["fit"]
    assert len(xr) == len(xm) and kr["epochs"] == km["epochs"] and kr["shuffle"] is False
    assert len(kr["validation_data"]) == len(km["validation_data"])
    cr = kr["callbacks"]
    assert [type(c).__name__ for c in cr] == [type(c).__name__ for c in cm]
    ck_r = cr[0].kwargs
    assert os.path.relpath(ck_r["filepath"], r["root"]) == os.path.relpath(cm[0].filepath, m["root"])
    assert (ck_r["monitor"], ck_r["save_weights_only"], ck_r["save_best_only"]) == \
        (cm[0].monitor, cm[0].save_weights_only, cm[0].save_best_only)
    assert cr[1].kwargs == {"monitor": cm[1].monitor, "patience": cm[1].patience}
    if scheduler == "sgdr":
        assert isinstance(cr[2], ref["SGDRC"]) and _numbers(cr[2]) == _numbers(cm[2])
        assert cr[3].args[0].__self__ is cr[2]                                                  # lr.lr_scheduler
    # evaluation: same report, same saved history
    assert r["report"] == m["report"]
    np.testing.assert_allclose(np.asarray(r["hist"][0], np.float64), np.asarray(m["hist"][0], np.float64), rtol=1e-12)
    np.testing.assert_allclose(np.asarray(r["hist"][1], np.float64), np.asarray(m["hist"][1], np.float64), rtol=0)
    assert r["hist"][2] == m["hist"][2]


@pytest.mark.parametrize("split,scaler,use_ring", [(True, True, False), (True, False, True), (False, True, True)])
def test_prepare_dataset_follows_the_reference(ref, tmp_path, split, scaler, use_ring):
    """``SCANN.prepare_dataset`` (scann_model.py:98-161) of the reference -- load_dataset, float32 mean / std target
    scaling, split_data, the three DataIterators -- beside ``scann_b200.model.SCANN.prepare_dataset`` on the same
    pickled data set and the same numpy seed: same split, same recorded config entries, bit-identical batches."""
    from scann_b200 import model as mine
    from tests.test_reference_pins import _batches, _write_dataset
    p_e, p_n = _write_dataset(tmp_path, n=61)
    out = {}
    for who, cls in (("mine", mine.SCANN), ("reference", ref and ref["SCANN"])):
        if cls is None:
            continue
        cfg = get_config("qm9")
        cfg["model"]["use_ring"] = use_ring
        cfg["hyper"].update(data_energy_path=p_e, data_nei_path=p_n, scaler=scaler, batch_size=8, test_percent=0.1,
                            train_size=None, test_size=None)
        obj = object.__new__(cls)
        obj.config, obj.mean, obj.std = cfg, 0, 1
        np.random.seed(23)
        if who == "reference":
            with ref["shim"].session({}, {}):
                res = obj.prepare_dataset(split=split)
        else:
            res = obj.prepare_dataset(split=split)
        out[who] = (obj, res)
    m, m_res = out["mine"]
    names = ("trainIter", "validIter", "testIter") if split else ("dataIter",)
    assert (m_res is None) == (not split)
    stored = {"mean_std": np.array([m.mean, m.std], np.float64), "mean_type": np.array(type(m.mean).__name__),
              "config": np.array([repr(m.config["hyper"][k]) for k in ("target_mean", "target_std", "data_size")])}
    for j, a in enumerate(m_res or ()):
        stored[f"split{j}"] = a
    for n in names:
        it = getattr(m, n)
        stored.update({f"{n}/{k}": v for k, v in _batches(it).items()})
        stored[f"{n}/shuffle_batch"] = np.array([it.shuffle, it.batch_size])
    check_stored(f"graph_prepare_dataset_{int(split)}{int(scaler)}{int(use_ring)}", stored)
    if ref is None:
        return
    r, r_res = out["reference"]
    assert r.mean == m.mean and r.std == m.std and type(r.mean) is type(m.mean)
    for k in ("target_mean", "target_std", "data_size"):
        assert r.config["hyper"][k] == m.config["hyper"][k], k
    if split:
        for a, b in zip(r_res, m_res):
            assert np.array_equal(a, b)
    else:
        assert r_res is None
    for n in names:
        a, b = getattr(r, n), getattr(m, n)
        assert len(a) == len(b) and a.shuffle == b.shuffle and a.batch_size == b.batch_size
        for i in range(len(a)):
            (ai, ae), (bi, be) = a[i], b[i]
            assert np.array_equal(ae, be) and ae.dtype == be.dtype and set(ai) == set(bi)
            for k in ai:
                assert ai[k].dtype == bi[k].dtype and np.array_equal(ai[k], bi[k]), (n, i, k)


def test_public_surface_matches_the_reference(ref):
    """Every public method of the reference's ``SCANN`` exists here with the same parameter names and defaults (extra
    optional parameters allowed), ``scann.layers`` exports the reference's ``__all__``, and the module-level helpers a
    reference user imports (``create_model``, ``DataIterator``, ``split_data`` ...) resolve under the same paths."""
    import importlib
    import inspect
    import json
    from scann_b200 import model as mine
    sigs = {name: [(p.name, repr(p.default)) for p in inspect.signature(f).parameters.values()]
            for name, f in inspect.getmembers(mine.SCANN, predicate=lambda x: inspect.isfunction(x) or inspect.ismethod(x))
            if not name.startswith("_") or name == "__init__"}
    check_stored("graph_public_surface", {"signatures": np.array(json.dumps(sigs, sort_keys=True))})
    theirs_methods = [] if ref is None else \
        inspect.getmembers(ref["SCANN"], predicate=lambda x: inspect.isfunction(x) or inspect.ismethod(x))
    for name, f in theirs_methods:
        if name.startswith("__") and name != "__init__":
            continue
        assert hasattr(mine.SCANN, name), name
        theirs = inspect.signature(f).parameters
        ours = inspect.signature(getattr(mine.SCANN, name)).parameters
        assert list(ours)[:len(theirs)] == list(theirs), name
        for p in theirs:
            assert ours[p].default == theirs[p].default or theirs[p].default is inspect.Parameter.empty, (name, p)
        for p in list(ours)[len(theirs):]:
            assert ours[p].default is not inspect.Parameter.empty, (name, p)       # extras must be optional
    ref_all = ["GlobalAttention", "LocalAttention", "ResidualNorm", "GaussianExpansion", "SGDRC",
               "root_mean_squared_error", "r2_square", "gather_shape", "mrelu"]      # scann/layers/__init__.py:7-17
    import scann.layers
    assert sorted(scann.layers.__all__) == sorted(ref_all)
    assert all(k in scann.layers._CUSTOM_OBJECTS for k in ref_all)
    for mod, names in {"scann.models": ["SCANN"], "scann.utils": ["DataIterator", "pad_sequence", "pad_nested_sequences",
                                                                 "split_data", "load_dataset"],
                       "scann.utils.general": ["pad_sequence", "pad_nested_sequences", "split_data", "load_dataset"],
                       "scann.utils.datagenerator": ["DataIterator"]}.items():
        m = importlib.import_module(mod)
        for n in names:
            assert hasattr(m, n), (mod, n)
    assert callable(mine.create_model)


def test_loss_and_metric_functions_match_the_reference(ref):
    """``root_mean_squared_error`` / ``r2_square`` (scann/layers/losses.py:5-16, the compile() loss and metric) of the
    reference against the host functions ``scann.layers`` exports here."""
    import scann.layers as L
    rng = np.random.default_rng(2)
    mine = np.zeros((3, 2))
    for j, n in enumerate((1, 7, 128)):
        yt, yp = rng.standard_normal((n, 1)), rng.standard_normal((n, 1))
        mine[j] = L.root_mean_squared_error(yt, yp), L.r2_square(yt, yp)
        if ref is None:
            continue
        with ref["shim"].session({}, {}):
            want_rmse = float(ref["root_mean_squared_error"](torch.tensor(yt), torch.tensor(yp)))
            want_r2 = float(ref["r2_square"](torch.tensor(yt), torch.tensor(yp)))
        assert abs(mine[j, 0] - want_rmse) <= 1e-14 * max(1.0, want_rmse)
        assert abs(mine[j, 1] - want_r2) <= 1e-12 * max(1.0, abs(want_r2))
    check_stored("graph_loss_metric", {"rmse_r2": mine}, rtol=1e-12, atol=1e-14)
