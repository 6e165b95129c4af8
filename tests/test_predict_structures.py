"""Structures in, predictions out on the device: ``voronoi.select_neighbors`` / ``neighbor_csr``
(``scann_voronoi_select`` + ``scann_voronoi_batch_csr``, csrc/voronoi.cu) and ``predict_structures``.

The host route they replace is ``compute_voronoi_neighbors`` -> ``DataIterator.csr_item`` -> ``predict``; the device
CSR must equal its arrays bit for bit, and the predictions must equal its predictions on the same padded shapes."""
import types

import numpy as np
import pytest

from tests.test_voronoi import _gpu_cases, molecule, random_cell, struct

PARAMS = [(4.0, 0.4), (6.0, 0.2), (8.0, 0.0)]


def hub(n=40, r=3.0, box=12.0):
    """An atom at the centre of n points on a sphere (Fibonacci lattice): its cell has n facets of similar size."""
    i = np.arange(n) + 0.5
    phi, th = np.arccos(1 - 2 * i / n), np.pi * (1 + 5 ** 0.5) * i
    P = r * np.stack([np.cos(th) * np.sin(phi), np.sin(th) * np.sin(phi), np.cos(phi)], -1)
    return struct(np.eye(3) * box, np.concatenate([[[0.0, 0.0, 0.0]], P]) + box / 2, [6] * (n + 1))


def lone_atom():
    """One site per 5 Angstrom cube: every facet at 5 Angstrom, none kept at d_t = 4."""
    return struct(np.eye(3) * 5.0, [[0.0, 0.0, 0.0]], [6])


def qm9_like(n, seed=0):
    rng = np.random.default_rng(seed)
    return [molecule(rng, int(rng.integers(9, 30))) for _ in range(n)]


def _data(structs, lists):
    de, dn = np.empty(len(structs), object), np.empty(len(structs), object)
    for k, (s, nb) in enumerate(zip(structs, lists)):
        de[k], dn[k] = (list(s.atomic_numbers), 0.0), nb
    return de, dn


def host_iterator(structs, d_t, w_t, angle, batch_size):
    from scann_b200 import voronoi as V
    from scann_b200.datagenerator import DataIterator
    de, dn = _data(structs, V.compute_voronoi_neighbors(structs, d_t, w_t))
    return DataIterator(de, dn, batch_size=batch_size, g_update=angle)


# ------------------------------------------------------------------------------------------------ CPU
def test_shape_classes():
    from scann_b200.model import shape_class
    assert shape_class(1, 0) == (8, 4)
    assert shape_class(29, 17) == (32, 20)
    assert shape_class(9, 32) == (16, 32)          # stays on the pipelined 32-row plan
    assert shape_class(64, 33) == (64, 40)
    assert shape_class(65, 60) == (72, 64)


def test_structure_chunks_keep_whole_batches():
    from scann_b200 import model as Mo
    n = [30] * 5000
    chunks = Mo._structure_chunks(n, 128)
    assert chunks[0][0] == 0 and chunks[-1][1] == 5000
    assert all(a == b for (_, a), (b, _) in zip(chunks, chunks[1:]))
    assert all(c0 % 128 == 0 for c0, _ in chunks)
    assert all(sum(n[c0:c1]) <= Mo._CHUNK_ATOMS for c0, c1 in chunks)
    assert Mo._structure_chunks([Mo._CHUNK_ATOMS] * 3, 2) == [(0, 2), (2, 3)]     # one batch may exceed the chunk


def test_new_entry_points_are_declared_and_bound():
    import os
    from scann_b200 import _abi
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                            "scann_b200.h")).read()
    for name in ("scann_voronoi_select", "scann_voronoi_batch_csr"):
        assert name in _abi.PROTOTYPES and f"int {name}(" in hdr


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def csr_cases():
    cases = [s for _, s in _gpu_cases()] + qm9_like(24, seed=7) + [hub(), lone_atom()]
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("angle", [True, False])
@pytest.mark.parametrize("d_t,w_t", PARAMS)
def test_device_csr_equals_the_data_iterator_bit_for_bit(csr_cases, d_t, w_t, angle):
    from scann_b200 import voronoi as V
    got = V.neighbor_csr(csr_cases, d_t, w_t, angle=angle)
    want, _ = host_iterator(csr_cases, d_t, w_t, angle, len(csr_cases)).csr_item(0)
    assert got["B"] == len(csr_cases) and got["M"] == want["M"] and got["N"] == want["N"]
    assert got["P"] == len(want["nbr_idx"])
    for key in ("struct_atom_off", "atom_nbr_off", "z", "nbr_idx"):
        assert np.array_equal(got[key].cpu().numpy(), np.asarray(want[key], np.int32)), key
    for key in ("nbr_w", "nbr_d"):
        assert np.array_equal(got[key].cpu().numpy().view(np.uint32), want[key].view(np.uint32)), key
    cnt = np.diff(want["atom_nbr_off"])
    assert np.array_equal(got["nmax"], [cnt[a:b].max(initial=0) for a, b in zip(want["struct_atom_off"][:-1],
                                                                            want["struct_atom_off"][1:])])
    hub_row = int(want["struct_atom_off"][-3])
    assert cnt.max() > 32 and cnt[hub_row] > 32                  # the hub's centre
    if d_t == 4.0:
        assert cnt[-1] == 0                                      # the lone atom keeps nothing


def _model(cfg_name, seed=3, n_attention=2, **over):
    from scann_b200.configs import get_config
    from scann_b200.model import create_model
    from scann_b200.config import model_spec
    from scann_b200.params import ParamLayout
    cfg = get_config(cfg_name)
    cfg["model"]["n_attention"] = n_attention
    cfg["model"].update(over)
    arena = ParamLayout(model_spec(cfg)).randomize_arena(seed)
    return create_model(cfg, infer=True, arena=arena), cfg


def host_predict(model, structs, d_t, w_t, angle, batch_size):
    """The host route on the same batches and padded shapes as predict_structures."""
    from scann_b200.model import shape_class
    it = host_iterator(structs, d_t, w_t, angle, batch_size)
    ys, gas = [], []
    for i in range(len(it)):
        csr, _ = it.csr_item(i)
        csr = dict(csr)
        csr["M"], csr["N"] = shape_class(csr["M"], csr["N"])
        y, ga = model.predict(csr)
        ys.append(y)
        gas.extend(ga[k, :n, 0] for k, n in enumerate(np.diff(csr["struct_atom_off"])))
    return np.concatenate(ys), gas


NOUP = {"g_update": False, "gaussian_d": 4.0, "use_ring": False}


@pytest.mark.gpu
@pytest.mark.parametrize("cfg_name,over", [("qm9", {}), ("ptgp", NOUP)], ids=["qm9_g_update", "ptgp_no_update"])
def test_predictions_equal_the_host_route_bit_for_bit(cfg_name, over):
    model, _ = _model(cfg_name, **over)
    structs = qm9_like(40, seed=11)
    structs[17:17] = [hub()]                                   # one batch with > 32 neighbours: the 64-row plan
    angle = bool(model.spec.g_update)
    y, ga = model.predict_structures(structs, batch_size=16)
    y_h, ga_h = host_predict(model, structs, 4.0, 0.4, angle, 16)
    assert np.array_equal(y, y_h)
    assert len(ga) == len(ga_h) and all(np.array_equal(a, b) for a, b in zip(ga, ga_h))
    eng = model.engine
    assert any(b.N > 32 for b in eng._batches.values()) and any(b.N <= 32 and b.stride == 32
                                                               for b in eng._batches.values())


@pytest.mark.gpu
def test_predictions_against_the_fp64_oracle():
    from oracle import scann_oracle as O
    from scann_b200 import voronoi as V
    from scann_b200.config import model_spec
    from scann_b200.datagenerator import prepare_input_from_neighbors
    from scann_b200.params import ParamLayout
    from tests.golden.make_golden import oracle_kwargs
    from tests.test_gpu_parity import TOL_OUT, rel
    model, cfg = _model("qm9")
    spec = model_spec(cfg)
    wd = ParamLayout(spec).to_dict(model.engine.get_params())
    rng = np.random.default_rng(8)
    structs = [molecule(rng, 12), molecule(rng, 21), random_cell(rng, 6), hub()]
    y, ga = model.predict_structures(structs)
    lists = V.compute_voronoi_neighbors(structs)
    for k, s in enumerate(structs):
        inp = prepare_input_from_neighbors(list(s.atomic_numbers), lists[k], angle=True)
        y_ref, ga_ref = O.predict(wd, inp, **oracle_kwargs(spec))
        assert rel(y[k], np.ravel(y_ref)) <= TOL_OUT and rel(ga[k], np.ravel(ga_ref)) <= TOL_OUT, k


@pytest.mark.gpu
def test_output_form_batch_size_and_scaling():
    from scann.models import SCANN
    from tests.test_gpu_parity import TOL_OUT, rel
    model, cfg = _model("qm9")
    assert model.spec.use_ga_norm
    structs = qm9_like(45, seed=5)
    y, ga = model.predict_structures(structs, batch_size=16)
    assert y.shape == (45, 1) and y.dtype == np.float32 and len(ga) == 45
    for s, g in zip(structs, ga):
        assert g.shape == (len(s.cart_coords),) and g.dtype == np.float32
        assert abs(float(g.sum(dtype=np.float64)) - 1.0) <= 1e-6
    y1, ga1 = model.predict_structures(structs[::-1][:5], batch_size=16)    # order follows the input
    assert np.array_equal(y1[:, 0], y[::-1][:5, 0]) or rel(y1[:, 0], y[::-1][:5, 0]) <= TOL_OUT
    for bs in (1, 7, 128):
        y2, ga2 = model.predict_structures(structs, batch_size=bs)
        assert rel(y2, y) <= TOL_OUT
        assert rel(np.concatenate(ga2), np.concatenate(ga)) <= TOL_OUT
    facade = SCANN.__new__(SCANN)
    facade.model, facade.mean, facade.std = model, 2.5, 4.0
    y3, ga3 = facade.predict_structures(structs, batch_size=16)
    assert np.array_equal(y3, y * np.float32(4.0) + 2.5) and all(np.array_equal(a, b) for a, b in zip(ga3, ga))
    y_d, _ = model.predict_structures(structs[:8], angle=False)            # angle picks the column
    y_t, _ = model.predict_structures(structs[:8], angle=True)
    assert np.array_equal(y_t, model.predict_structures(structs[:8])[0]) and not np.array_equal(y_d, y_t)


@pytest.mark.gpu
def test_errors_name_the_caller_index_and_leave_the_device_usable():
    model, _ = _model("qm9")
    good = qm9_like(9, seed=2)
    before, _ = model.predict_structures(good, batch_size=4)
    bad = struct(np.eye(3) * 10.0, [[1, 1, 1], [2, 2, 2], [2, 2, 2 + 1e-10]], [6, 6, 6])
    with pytest.raises(ValueError, match=r"^structure 6, site 1: two points"):
        model.predict_structures(good[:6] + [bad] + good[6:], batch_size=4)
    with pytest.raises(ValueError, match=r"structure 2 has no lattice"):
        model.predict_structures(good[:2] + [types.SimpleNamespace(cart_coords=np.zeros((2, 3)), lattice=None,
                                                                    atomic_numbers=(6, 6))])
    big = struct(np.eye(3) * 200.0, np.random.default_rng(0).random((1001, 3)) * 200.0, [6] * 1001)
    with pytest.raises(ValueError, match=r"structure 1 has 1001 sites"):
        model.predict_structures([good[0], big])
    after, _ = model.predict_structures(good, batch_size=4)
    assert np.array_equal(before, after)
    ring, _ = _model("ptgp", g_update=False, gaussian_d=4.0)
    with pytest.raises(NotImplementedError, match="use_ring"):
        ring.predict_structures(good)
    from scann_b200.config import model_spec
    from scann_b200.configs import get_config
    from scann_b200.model import ScannKerasModel
    cfg = get_config("qm9", feature="cgcnn")
    cfg["model"]["n_attention"] = 1
    with pytest.raises(NotImplementedError, match="cgcnn"):
        ScannKerasModel(model_spec(cfg), infer=True).predict_structures(good)


@pytest.mark.gpu
def test_a_thousand_molecules_stay_within_the_shape_class_cache():
    model, _ = _model("qm9")
    eng = model.engine
    structs = qm9_like(1000, seed=21)
    y, ga = model.predict_structures(structs, batch_size=128)
    assert len(ga) == 1000 and np.isfinite(y).all()
    assert eng.shape_class_evictions == 0
    assert eng.graph_captures == len(eng._batches) <= eng.max_shape_classes, sorted(eng._batches)
    n0 = eng.graph_captures
    model.predict_structures(structs, batch_size=128)          # a second pass replays every graph
    assert eng.graph_captures == n0 and eng.shape_class_evictions == 0
