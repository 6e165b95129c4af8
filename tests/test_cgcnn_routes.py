"""``feature='cgcnn'`` models on the batches that carry atomic numbers: CSR batches (``predict`` on
``DataIterator.csr_item``), ``predict_structures`` and ``DeviceDataIterator`` (``fit``, ``evaluate``).

embed_atom of a cgcnn model is ``Dense(92 -> E)`` applied to ``table[Z]``, so its output for an atom is row Z of
``emb_table = table @ W + b`` (one small launch per forward), and its gradients follow from the per-element sums of the
embedding backward through ``scann_cgcnn_table_backward``.  The forward is bit-identical to the padded feature-vector
route; the gradients sum in another order and agree with it, and with the fp64 oracle, within the parity tolerance."""
import ctypes
import types

import numpy as np
import pytest

from tests.test_device_data import ragged_set
from tests.test_predict_structures import hub, qm9_like
from tests.test_voronoi import random_cell, struct

ROUTE = "atomic_features"


def table(n=100):
    from scann_b200.synth import cgcnn_table
    return cgcnn_table(n)


def cgcnn_iterator(de, dn, T, **kw):
    from scann_b200.datagenerator import DataIterator
    return DataIterator(de, dn, feature="cgcnn", atomic_features=T, **kw)


# ------------------------------------------------------------------------------------------------ CPU
def test_table_validation():
    from scann_b200.datagenerator import check_atomic_features
    T = table()
    assert check_atomic_features(T) is not None and check_atomic_features(T).shape == (100, 92)
    assert np.array_equal(check_atomic_features({"0": [0.0] * 92, "2": [1.0] * 92})[2], np.ones(92, np.float32))
    assert check_atomic_features(T[:1]).shape == (1, 92)              # the padding row alone
    bad = T.copy()
    bad[7, 3] = np.nan
    for t, msg in [(T.astype(np.float64), "float32"), (T[:, :91], r"\[Z \+ 1, 92\]"), (T[0], r"\[Z \+ 1, 92\]"),
                   (T[:0], r"\[Z \+ 1, 92\]"), (bad, "row 7"), (np.where(T > 0, np.inf, T).astype(np.float32), "row")]:
        with pytest.raises(ValueError, match=msg):
            check_atomic_features(t)


def test_table_backward_refuses_bad_sizes():
    from scann_b200 import _abi
    for Z, F, E in [(10, 91, 64), (10, 92, 0), (10, 92, 129), (0, 92, 64)]:
        assert _abi.lib.scann_cgcnn_table_backward(None, None, Z, F, E, None, None, None) != 0
        assert "cgcnn_table_backward: bad sizes" in _abi.last_error()


def test_an_unknown_element_names_the_structure():
    from scann_b200.datagenerator import DeviceDataIterator, check_table_rows
    check_table_rows(np.array([1, 6, 99]), np.array([0, 2, 3]), 100)
    with pytest.raises(ValueError, match=r"structure 1: atomic number 100 has no row .*100 rows"):
        check_table_rows(np.array([1, 6, 100]), np.array([0, 2, 3]), 100)
    de, dn = ragged_set(20, seed=3)
    it = cgcnn_iterator(de, dn, table(), batch_size=8)
    assert it.atomic_features is not None and it.atomic_features.shape == (100, 92)
    it.atomic_features = table(9)                 # Z up to 9: the fluorine atoms have no row
    s = int(np.searchsorted(it.atom_off, int(np.argmax(it.z == 9)), side="right")) - 1
    with pytest.raises(ValueError, match=f"structure {s}: atomic number 9 has no row"):
        DeviceDataIterator.from_data_iterator(it)
    ok = struct(np.eye(3) * 5.0, [[0.0, 0.0, 0.0]], [6])
    heavy = struct(np.eye(3) * 5.0, [[0.0, 0.0, 0.0], [2.5, 2.5, 2.5]], [6, 118])
    with pytest.raises(ValueError, match="structure 2: atomic number 118 has no row"):
        DeviceDataIterator.from_structures([ok, ok, heavy], [0.0] * 3, feature="cgcnn", atomic_features=table())


def test_refusals_without_a_table_say_how_to_pass_one():
    from scann_b200.datagenerator import DeviceDataIterator as D
    msg = r"feature='cgcnn'.*atomic_features="
    with pytest.raises(NotImplementedError, match=msg):
        D.from_data_iterator(types.SimpleNamespace(feature="cgcnn", atomic_features=None))
    with pytest.raises(NotImplementedError, match=msg):
        D.from_structures([], [], feature="cgcnn")
    de, dn = ragged_set(10)
    it = cgcnn_iterator(de, dn, table(), batch_size=4)
    pair_off, nmax, npairs = D.host_sizes(it.atom_off, it.nbr_off, it.nbr_idx)
    with pytest.raises(NotImplementedError, match=msg):
        D({}, it.energy, it.atom_off, pair_off, nmax, npairs, feature="cgcnn")
    with pytest.raises(NotImplementedError, match="use_ring.*openbabel"):     # unchanged
        D.from_structures([], [], use_ring=True, feature="cgcnn", atomic_features=table())


def test_padded_items_equal_the_data_iterator():
    """DeviceDataIterator.__getitem__ of a cgcnn data set: the gathered batch (here packed on the host from the same
    CSR slice) with the atomic numbers replaced through the iterator's own table, as DataIterator does."""
    from scann_b200.datagenerator import DeviceDataIterator, pack_padded
    de, dn = ragged_set(50, seed=4, use_ring=True)
    T = table()
    T[0] = 0.5                                  # padded atoms read row 0
    np.random.seed(5)
    host = cgcnn_iterator(de, dn, T, batch_size=16, shuffle=True, use_ring=True)
    dev = DeviceDataIterator({}, host.energy, host.atom_off, *DeviceDataIterator.host_sizes(host.atom_off, host.nbr_off,
                                                                                            host.nbr_idx),
                             batch_size=16, shuffle=True, use_ring=True, indexes=host.indexes, feature="cgcnn",
                             atomic_features=host.atomic_features)
    assert dev.feature == "cgcnn" and np.array_equal(dev.atomic_features, T)

    def gathered(i):
        csr, e = host.csr_item(i)
        return pack_padded(csr), e
    dev._gathered_item = gathered
    for i in range(len(host)):
        (ih, th), (id_, td) = host[i], dev[i]
        assert ih.keys() == id_.keys() and np.array_equal(th, td)
        assert id_["atomic"].shape[-1] == 92 and (id_["atomic"][~id_["atom_mask"][..., 0]] == 0.5).all()
        for k in ih:
            assert ih[k].dtype == id_[k].dtype and np.array_equal(ih[k], id_[k]), (i, k)


# ------------------------------------------------------------------------------------------------ GPU
def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


@pytest.mark.gpu
@pytest.mark.parametrize("Z", [1, 33, 101])
@pytest.mark.parametrize("E", [48, 128])
def test_table_backward_kernel_against_float64(Z, E):
    import torch
    from scann_b200 import _abi
    rng = np.random.default_rng(Z * 1000 + E)
    T = rng.standard_normal((Z, 92)).astype(np.float32)
    dE = rng.standard_normal((Z, E)).astype(np.float32)
    W0 = rng.standard_normal((92, E)).astype(np.float32)
    b0 = rng.standard_normal(E).astype(np.float32)
    want_W = W0.astype(np.float64) + T.astype(np.float64).T @ dE.astype(np.float64)
    want_b = b0.astype(np.float64) + dE.astype(np.float64).sum(0)
    dev = [torch.from_numpy(a).cuda() for a in (T, dE)]
    outs = []
    for _ in range(2):
        dW, db = torch.from_numpy(W0).cuda(), torch.from_numpy(b0).cuda()
        st = torch.cuda.current_stream().cuda_stream
        _abi.check(_abi.lib.scann_cgcnn_table_backward(_ptr(dev[0]), _ptr(dev[1]), Z, 92, E, _ptr(dW), _ptr(db), st))
        torch.cuda.synchronize()
        outs.append((dW.cpu().numpy(), db.cpu().numpy()))
    for got, want in ((outs[0][0], want_W), (outs[0][1], want_b)):
        assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max()
    assert all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(outs[0], outs[1]))


def _cg_model(cfg_name="qm9", L=2, seed=3, infer=True, deterministic=None, **over):
    from scann_b200.config import model_spec
    from scann_b200.configs import get_config
    from scann_b200.model import create_model
    from scann_b200.params import ParamLayout
    cfg = get_config(cfg_name, feature="cgcnn")
    cfg["model"]["n_attention"] = L
    cfg["model"].update(over)
    arena = ParamLayout(model_spec(cfg)).randomize_arena(seed)
    return create_model(cfg, infer=infer, arena=arena, deterministic=deterministic), cfg


def mp_like(n, seed=0):
    rng = np.random.default_rng(seed)
    cells = [random_cell(rng, int(rng.integers(2, 17))) for _ in range(n)]
    return [struct(c.lattice.matrix, c.cart_coords, rng.integers(1, 95, len(c.cart_coords))) for c in cells]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg_name", ["qm9", "mp2018"])
def test_predict_structures_equals_padded_feature_batches(cfg_name):
    """Bit equality with predict on padded DataIterator(feature='cgcnn') batches of the same structures in the same
    shape classes (y, ga, every layer's scores), and the fp64 oracle within TOL_OUT."""
    import torch
    from oracle import scann_oracle as O
    from scann_b200 import voronoi as V
    from scann_b200.datagenerator import pack_padded, prepare_input_from_neighbors
    from scann_b200.model import shape_class
    from scann_b200.params import ParamLayout
    from tests.golden.make_golden import oracle_kwargs
    from tests.test_gpu_parity import TOL_OUT, rel
    from tests.test_predict_structures import _data
    model, _ = _cg_model(cfg_name)
    spec = model.spec
    T = table()
    T[0] = 0.25
    structs = qm9_like(30, seed=11) if cfg_name == "qm9" else mp_like(30, seed=11)
    structs[9:9] = [hub()]                                 # one batch with > 32 neighbours: the 64-row plan
    angle = bool(spec.g_update)
    y, ga, la = model.predict_structures(structs, batch_size=16, local_attention=True, atomic_features=T)
    lists = V.compute_voronoi_neighbors(structs)
    de, dn = _data(structs, lists)
    it = cgcnn_iterator(de, dn, T, batch_size=16, g_update=angle)
    k = 0
    for i in range(len(it)):
        csr, _ = it.csr_item(i)
        csr = dict(csr)
        csr["M"], csr["N"] = shape_class(csr["M"], csr["N"])
        inputs = pack_padded(csr)
        inputs["atomic"] = T[inputs["atomic"]]             # DataIterator.__getitem__ on the shape class
        y_h, ga_h, la_h = model.predict(inputs, local_attention=True)
        sa, an = csr["struct_atom_off"], csr["atom_nbr_off"]
        for s in range(len(sa) - 1):
            n = sa[s + 1] - sa[s]
            assert y[k, 0].view(np.uint32) == y_h[s, 0].view(np.uint32), k
            assert np.array_equal(ga[k].view(np.uint32), ga_h[s, :n, 0].view(np.uint32)), k
            cols = [la_h[:, s, :, m, :an[sa[s] + m + 1] - an[sa[s] + m]] for m in range(n)]
            assert np.array_equal(la[k].scores.view(np.uint32), np.concatenate(cols, axis=2).view(np.uint32)), k
            k += 1
    assert k == len(structs)
    assert any(b.N > 32 for b in model.engine._batches.values())
    wd = ParamLayout(spec).to_dict(model.engine.get_params())
    for k in (0, 9, 20):
        inp = prepare_input_from_neighbors(list(structs[k].atomic_numbers), lists[k], angle=angle)
        inp["atomic"] = T[inp["atomic"]]
        y_ref, ga_ref = O.predict(wd, inp, **oracle_kwargs(spec))
        # a single output of a cancelling sum: bounded by TOL_OUT or 5 x the distance of the reference's own fp32
        # arithmetic (fp32 oracle) from fp64, as the golden cases are (tests/test_gpu_parity.py golden_y_tolerance)
        y32, _ = O.predict(wd, inp, torch.float32, **oracle_kwargs(spec))
        tol_y = max(TOL_OUT, 5.0 * rel(np.ravel(y32), np.ravel(y_ref)))
        assert rel(y[k], np.ravel(y_ref)) <= tol_y and rel(ga[k], np.ravel(ga_ref)) <= TOL_OUT, k
    with pytest.raises(NotImplementedError, match=r"atomic_features="):
        _cg_model(cfg_name)[0].predict_structures(structs[:2])


@pytest.mark.gpu
def test_predict_on_csr_batches_needs_the_table_then_equals_the_padded_batch():
    model, _ = _cg_model()
    de, dn = ragged_set(40, seed=6)
    T = table()
    it = cgcnn_iterator(de, dn, T, batch_size=16)
    first = model.predict(it[0][0])                    # the padded route fills the shape class's feature buffer
    with pytest.raises(ValueError, match="atomic_features"):
        model.predict(it.csr_item(0)[0])
    model.engine.set_atomic_features(T)
    for i in range(len(it)):
        y_p, ga_p = model.predict(it[i][0])
        y_c, ga_c = model.predict(it.csr_item(i)[0])
        assert np.array_equal(y_p.view(np.uint32), y_c.view(np.uint32)), i
        assert np.array_equal(ga_p.view(np.uint32), ga_c.view(np.uint32)), i
    assert np.array_equal(first[0], model.predict(it[0][0])[0])


def _grads(eng):
    import torch
    torch.cuda.synchronize()
    eng.check_status()
    return eng.layout.to_dict(eng.grad_out.cpu().numpy())


@pytest.mark.gpu
@pytest.mark.parametrize("over,ring", [({}, False), ({"g_update": False, "gaussian_d": 4.0}, False), ({}, True)],
                         ids=["g_update", "no_update", "ring"])
def test_gradients_of_a_gathered_batch_against_the_oracle(over, ring):
    import torch
    from oracle import scann_oracle as O
    from scann_b200.datagenerator import DeviceDataIterator
    from scann_b200.engine import Engine
    from tests.golden.make_golden import oracle_kwargs
    from tests.test_gpu_parity import TOL_GRAD
    model, _ = _cg_model(infer=False, seed=13, use_ring=ring, **over)
    spec = model.spec
    arena = model.engine.get_params()
    lay = model.layout
    de, dn = ragged_set(12, seed=9, use_ring=ring)
    T = table()
    T[0] = 0.5
    dev = DeviceDataIterator.from_data_iterator(cgcnn_iterator(de, dn, T, batch_size=6, use_ring=ring,
                                                               g_update=spec.g_update))
    eng = model.engine
    eng.set_atomic_features(dev.atomic_features)
    b = eng.load_batch_gather(dev, *dev.batch_shape(0), plan=False)
    assert b.route == ROUTE
    eng.train_step(b, b.target, lr=1e-3, apply=False, want_grads=True, replan=True)
    g = _grads(eng)
    inputs, target = dev[0]
    w = lay.to_dict(arena)
    loss, _, _, ref = O.loss_and_grads(w, inputs, target, [e.name for e in lay if e.l2], use_ring=spec.use_ring,
                                       **oracle_kwargs(spec))
    gmax = max(np.abs(v).max() for v in ref.values())
    padded = Engine(spec, arena)                         # the padded feature-vector route of the same batch
    bp = padded.load_batch(inputs)
    padded.train_step(bp, torch.from_numpy(target).cuda(), lr=1e-3, apply=False, want_grads=True)
    gp = _grads(padded)
    for e in lay:
        bound = TOL_GRAD * max(np.abs(ref[e.name]).max(), 1e-3 * gmax)
        assert np.abs(g[e.name].astype(np.float64) - ref[e.name]).max() <= bound, e.name
        assert np.abs(g[e.name].astype(np.float64) - gp[e.name]).max() <= bound, e.name
    assert np.abs(g["embed_atom/kernel"]).max() > 0 and np.abs(g["embed_atom/bias"]).max() > 0
    lv = eng.loss_value(b.B).cpu().numpy()
    assert abs(lv[0] - float(loss)) <= 1e-5 * abs(float(loss))


def _fit_device(de, dn, T):
    from scann_b200.datagenerator import DeviceDataIterator
    np.random.seed(21)
    it = cgcnn_iterator(de[:160], dn[:160], T, batch_size=32, shuffle=True, g_update=True)
    vit = cgcnn_iterator(de[160:], dn[160:], T, batch_size=32, g_update=True)
    it, vit = DeviceDataIterator.from_data_iterator(it), DeviceDataIterator.from_data_iterator(vit)
    m, _ = _cg_model(infer=False, seed=4, deterministic=True)
    m.compile(optimizer=5e-4)
    hist = m.fit(it, epochs=2, validation_data=vit, verbose=0)
    eng = m.engine
    assert eng.train_dropout and eng.deterministic
    return {"hist": hist.history, "params": eng.params.cpu().numpy(), "m": eng.adam_m.cpu().numpy(),
            "v": eng.adam_v.cpu().numpy()}


@pytest.mark.gpu
def test_deterministic_fit_over_the_device_route_repeats_its_bits():
    de, dn = ragged_set(200, seed=8)
    T = table()
    a, b = _fit_device(de, dn, T), _fit_device(de, dn, T)
    assert a["hist"] == b["hist"] and len(a["hist"]["val_mae"]) == 2
    for k in ("params", "m", "v"):
        assert np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)), k


@pytest.mark.gpu
def test_padded_and_table_routes_keep_separate_graphs():
    from scann_b200.datagenerator import DeviceDataIterator
    de, dn = ragged_set(40, seed=6)
    T = table()
    it = cgcnn_iterator(de, dn, T, batch_size=40)             # one batch: one shape class
    dev = DeviceDataIterator.from_data_iterator(it)

    def padded_steps(m):
        m.predict(it[0][0])
        m.train_on_batch(*it[0])
        m.predict(it[0][0])
        m.train_on_batch(*it[0])
        (b,) = m.engine._batches.values()
        return b, {k: g.n_launches for k, g in b.graphs.items()}

    ref, _ = _cg_model(infer=False)
    _, want = padded_steps(ref)                          # an engine that never sees a table
    assert sorted(want) == [("infer", True), ("train", True, True, False, False)]
    m, _ = _cg_model(infer=False)
    m.predict_device_batch(dev, 0)
    m.fit(dev, epochs=1, verbose=0)
    b, got = padded_steps(m)
    assert len(m.engine._batches) == 1                  # one shape class, both routes
    assert sorted(got) == sorted(list(want) + [("infer", True, ROUTE), ("train", True, True, False, False, ROUTE)])
    assert all(got[k] == want[k] for k in want)
    n = m.engine.graph_captures
    m.engine.set_atomic_features(T.copy())              # same shape, same values: graphs stay
    m.engine.set_atomic_features(np.ascontiguousarray(T[::-1]))          # same shape, new values: copied in place
    m.predict_device_batch(dev, 0)
    assert m.engine.graph_captures == n
    m.engine.set_atomic_features(table(120))             # another row count: the table route's graphs are dropped
    assert sorted(b.graphs) == sorted(want)
    m.predict_device_batch(dev, 0)
    assert m.engine.graph_captures == n + 1


@pytest.mark.gpu
def test_a_thousand_molecules_stay_within_the_shape_class_cache():
    model, _ = _cg_model()
    eng = model.engine
    structs = qm9_like(1000, seed=21)
    y, ga = model.predict_structures(structs, batch_size=128, atomic_features=table())
    assert len(ga) == 1000 and np.isfinite(y).all()
    assert eng.shape_class_evictions == 0
    assert eng.graph_captures == len(eng._batches) <= eng.max_shape_classes, sorted(eng._batches)
