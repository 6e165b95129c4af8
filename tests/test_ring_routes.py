"""``use_ring`` models on the structure routes: ``predict_structures``, ``DeviceDataIterator.from_structures`` and
``SCANN.prepare_structures`` take the ring / aromatic flags as ``ring_aromatic=`` (one ``[n_sites, 2]`` integer array
per structure, the third item of a reference ``data_energy`` row).

The flags are not a function of the geometry (openbabel perceives them from bonds), so these routes cannot make them:
the caller passes them and the routes refuse a ring model without them.  On the device they travel as the ``ring``
segment of a CSR blob (``NeighborSelection.csr(..., ring=)``) or the ``ring`` array of a ``DeviceDataIterator``, which
``scann_pack_batch`` / ``scann_gather_batch`` read as on the host CSR route; the outputs, buffers and training bits
must be those of ``DataIterator(..., use_ring=True)`` batches of the same structures."""
import os

import numpy as np
import pytest

from tests.test_predict_structures import hub, qm9_like
from tests.test_voronoi import struct

CC = 1.42                                           # C-C bond of graphene, Angstrom
PT_NN = 2.77                                        # Pt-Pt nearest-neighbour distance (fcc, a = 3.92 Angstrom)
SHEETS = [(7, 6), (8, 6), (7, 7), (9, 6), (8, 7), (10, 6)]      # rectangular graphene cells: 168 .. 240 carbons


def _pt_sites():
    """fcc sites (nearest neighbours PT_NN apart) on and above the plane z = 0, nearest the origin first."""
    g = np.arange(-2, 3)
    p = np.array([(i, j, k) for i in g for j in g for k in range(3) if (i + j + k) % 2 == 0], np.float64)
    p = p[np.lexsort((p[:, 1], p[:, 0], p[:, 2], np.round(np.linalg.norm(p, axis=1), 9)))]
    return p * PT_NN / np.sqrt(2)


def ptgp_like(n, seed=0):
    """PtGP-like structures: a periodic graphene sheet (C-C 1.42 Angstrom, positions jittered by 0.02 Angstrom, 10
    Angstrom cell along c) with a Pt cluster of 4-13 atoms 2.3 Angstrom above it, 172-253 sites.  Returns the
    structures and their ring / aromatic flags: carbon [1, 1] and Pt [0, 0] (the pattern of the data set), replaced
    by random integers in every third structure so that no test rests on one pattern.

    A Pt atom with fewer cluster neighbours meets the carbons of both sheets across the vacuum: the Voronoi cell of a
    lone adatom has 60-86 facets (scipy oracle, cells 8-14 Angstrom high), beyond the cell search's capacity of 64.
    Clusters from 4 atoms in a 10 Angstrom cell mostly stay within it: the structures of these tests have at most 56
    facets per cell, while a few in a hundred larger draws do not."""
    rng = np.random.default_rng(seed)
    a, b = np.sqrt(3) * CC, 3 * CC
    cell = np.array([[0, 0], [a / 2, CC / 2], [a / 2, 1.5 * CC], [0, 2 * CC]])
    pt = _pt_sites()
    structs, flags = [], []
    for k in range(n):
        nx, ny = SHEETS[int(rng.integers(len(SHEETS)))]
        L = np.diag([nx * a, ny * b, 10.0])
        xy = (cell[None, None] + np.stack(np.meshgrid(np.arange(nx) * a, np.arange(ny) * b, indexing="ij"),
                                          -1)[:, :, None]).reshape(-1, 2)
        C = np.concatenate([xy, np.full((len(xy), 1), 3.0)], 1) + rng.normal(0, 0.02, (len(xy), 3))
        m = int(rng.integers(4, 14))
        th = rng.uniform(0, 2 * np.pi)
        rot = np.array([[np.cos(th), -np.sin(th), 0], [np.sin(th), np.cos(th), 0], [0, 0, 1]])
        P = pt[:m] @ rot.T + [rng.uniform(0, L[0, 0]), rng.uniform(0, L[1, 1]), 3.0 + 2.3]
        X = np.concatenate([C, P])
        structs.append(struct(L, X % np.diag(L), [6] * len(C) + [78] * m))
        f = np.concatenate([np.ones((len(C), 2), np.int64), np.zeros((m, 2), np.int64)])
        flags.append(rng.integers(-3, 4, f.shape) if k % 3 == 2 else f)
    return structs, flags


def random_flags(structs, seed=0):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 2, (len(s.atomic_numbers), 2)) for s in structs]


def ring_rows(structs, lists, flags, targets=None):
    """``data_energy`` / ``data_neighbor`` of the reference with the flags as the third item of each row."""
    de, dn = np.empty(len(structs), object), np.empty(len(structs), object)
    for k, (s, nb) in enumerate(zip(structs, lists)):
        de[k] = (list(s.atomic_numbers), 0.0 if targets is None else targets[k], np.asarray(flags[k]).tolist())
        dn[k] = nb
    return de, dn


def _ring_model(cfg_name, seed=3, infer=True, feature="atomic", deterministic=None, **over):
    from scann_b200.config import model_spec
    from scann_b200.configs import get_config
    from scann_b200.model import create_model
    from scann_b200.params import ParamLayout
    cfg = get_config(cfg_name, feature=feature)
    cfg["model"].update(use_ring=True, **over)
    arena = ParamLayout(model_spec(cfg)).randomize_arena(seed)
    return create_model(cfg, infer=infer, arena=arena, deterministic=deterministic), cfg


PTGP = {"g_update": False, "gaussian_d": 4.0}       # the shipped yaml lacks both keys (configs.py)


# ------------------------------------------------------------------------------------------------ CPU
def test_generator_makes_ptgp_sized_structures():
    structs, flags = ptgp_like(12, seed=1)
    for s, f in zip(structs, flags):
        n = len(s.atomic_numbers)
        assert 150 <= n <= 256 and f.shape == (n, 2)
        X = np.asarray(s.cart_coords)
        L = np.diag(s.lattice.matrix)
        d = X[:, None] - X[None]
        d -= np.round(d / L) * L
        r = np.linalg.norm(d, axis=-1) + np.eye(n) * 9
        assert r.min() > 1.2                          # no two sites closer than a bond
    assert any(len(s.atomic_numbers) > 193 for s in structs)


def test_check_ring_aromatic_takes_the_forms_of_a_data_energy_row():
    from scann_b200.datagenerator import check_ring_aromatic
    flags = [[[1, 0], [0, 1]], np.array([[2, 3]], np.int64), np.array([[True, False]] * 3),
             np.array([[1.0, -4.0]], np.float32), np.zeros((0, 2), np.uint8), np.array([[-2 ** 31, 2 ** 31 - 1]])]
    got = check_ring_aromatic(flags, [2, 1, 3, 1, 0, 1])
    assert got.dtype == np.int32 and got.flags.c_contiguous and got.shape == (8, 2)
    assert got.tolist() == [[1, 0], [0, 1], [2, 3], [1, 0], [1, 0], [1, 0], [1, -4], [-2 ** 31, 2 ** 31 - 1]]
    assert check_ring_aromatic([], []).shape == (0, 2)


@pytest.mark.parametrize("bad,msg", [
    (np.ones((3, 3), np.int32), r"structure 2: ring_aromatic must be \[3, 2\] \(one row per site\), not \[3, 3\]"),
    (np.ones((2, 2), np.int32), r"structure 2: .*\[3, 2\].*not \[2, 2\]"),
    (np.ones(6, np.int32), r"structure 2: .*not \[6\]"),
    (np.full((3, 2), 0.5), "structure 2: ring_aromatic holds a value that is not an integer"),
    (np.full((3, 2), np.nan), "structure 2: .*not an integer"),
    (np.full((3, 2), 2 ** 31), "structure 2: ring_aromatic holds a value outside int32"),
    (np.full((3, 2), -2 ** 31 - 1), "structure 2: .*outside int32"),
    (np.full((3, 2), 2.0 ** 40), "structure 2: .*outside int32"),
    (np.full((3, 2), "1"), "structure 2: ring_aromatic must hold integers"),
    (np.full((3, 2), None), "structure 2: ring_aromatic must hold integers"),
])
def test_check_ring_aromatic_names_the_structure(bad, msg):
    from scann_b200.datagenerator import check_ring_aromatic
    ok = np.zeros((2, 2), np.int32)
    with pytest.raises(ValueError, match=msg):
        check_ring_aromatic([ok, ok, bad, ok], [2, 2, 3, 2])


def test_check_ring_aromatic_counts_the_arrays():
    from scann_b200.datagenerator import check_ring_aromatic
    with pytest.raises(ValueError, match="3 structures but 2 ring_aromatic arrays"):
        check_ring_aromatic([np.zeros((1, 2))] * 2, [1, 1, 1])
    with pytest.raises(ValueError, match="sequence of"):
        check_ring_aromatic(5, [1])


def _three():
    ok = struct(np.eye(3) * 5.0, [[0.0, 0.0, 0.0]], [6])
    two = struct(np.eye(3) * 6.0, [[0.0, 0.0, 0.0], [3.0, 3.0, 3.0]], [6, 8])
    return [ok, two, two], [np.ones((1, 2), int), np.ones((2, 2), int), np.ones((2, 2), int)]


RING_REFUSAL = r"use_ring.*openbabel.*ring_aromatic="


def test_from_structures_refusals_and_checks():
    from scann_b200.datagenerator import DeviceDataIterator as D
    structs, flags = _three()
    with pytest.raises(NotImplementedError, match=RING_REFUSAL):
        D.from_structures(structs, [0.0] * 3, use_ring=True)
    with pytest.raises(ValueError, match="ring_aromatic is read by use_ring models only"):
        D.from_structures(structs, [0.0] * 3, ring_aromatic=flags)
    with pytest.raises(ValueError, match="3 structures but 2 ring_aromatic arrays"):
        D.from_structures(structs, [0.0] * 3, use_ring=True, ring_aromatic=flags[:2])
    with pytest.raises(ValueError, match=r"structure 2: .*\[2, 2\].*not \[1, 2\]"):
        D.from_structures(structs, [0.0] * 3, use_ring=True, ring_aromatic=flags[:2] + [flags[0]])
    with pytest.raises(NotImplementedError, match="use_ring.*openbabel"):     # the cgcnn table does not stand in
        D.from_structures([], [], use_ring=True, feature="cgcnn",
                          atomic_features=np.zeros((10, 92), np.float32))


def _bare_model(use_ring, feature="atomic"):
    """A ScannKerasModel with its spec only: every check of predict_structures runs before the engine is used."""
    from scann_b200.config import model_spec
    from scann_b200.configs import get_config
    from scann_b200.model import ScannKerasModel
    cfg = get_config("qm9", feature=feature)
    cfg["model"].update(n_attention=1, use_ring=use_ring)
    m = ScannKerasModel.__new__(ScannKerasModel)
    m.spec = model_spec(cfg)
    return m


def test_predict_structures_refusals_and_checks_across_chunks(monkeypatch):
    from scann_b200 import model as Mo
    structs = qm9_like(10, seed=4)
    flags = random_flags(structs)
    with pytest.raises(NotImplementedError, match=RING_REFUSAL):
        _bare_model(True).predict_structures(structs)
    with pytest.raises(NotImplementedError, match=RING_REFUSAL):
        _bare_model(True, "cgcnn").predict_structures(structs, atomic_features=np.zeros((10, 92), np.float32))
    with pytest.raises(ValueError, match="ring_aromatic is read by use_ring models only"):
        _bare_model(False).predict_structures(structs, ring_aromatic=flags)
    monkeypatch.setattr(Mo, "_CHUNK_ATOMS", 60)              # several chunks of two-structure batches
    assert len(Mo._structure_chunks([len(s.atomic_numbers) for s in structs], 2)) > 2
    bad = list(flags)
    bad[7] = np.full_like(flags[7], 2 ** 31)
    with pytest.raises(ValueError, match="structure 7: ring_aromatic holds a value outside int32"):
        _bare_model(True).predict_structures(structs, batch_size=2, ring_aromatic=bad)
    with pytest.raises(ValueError, match="10 structures but 9 ring_aromatic arrays"):
        _bare_model(True).predict_structures(structs, batch_size=2, ring_aromatic=flags[:9])


def _bare_scann(use_ring):
    from scann.models import SCANN
    from scann_b200.configs import get_config
    s = SCANN.__new__(SCANN)
    s.config = get_config("qm9")
    s.config["model"].update(n_attention=1, use_ring=use_ring)
    s.config["hyper"].update(test_percent=0.25, train_size=None, test_size=None)
    return s


def test_prepare_structures_refusals_and_checks_name_the_callers_index():
    structs = qm9_like(8, seed=5)
    flags = random_flags(structs)
    with pytest.raises(NotImplementedError, match=RING_REFUSAL):
        _bare_scann(True).prepare_structures(structs, [0.0] * 8)
    with pytest.raises(ValueError, match="ring_aromatic is read by use_ring models only"):
        _bare_scann(False).prepare_structures(structs, [0.0] * 8, ring_aromatic=flags)
    bad = list(flags)
    bad[5] = flags[5][:-1]
    s = _bare_scann(True)
    with pytest.raises(ValueError, match=r"structure 5: ring_aromatic must be \[\d+, 2\]"):
        s.prepare_structures(structs, [0.0] * 8, ring_aromatic=bad)
    assert "data_size" not in s.config["hyper"]             # refused before the targets are scaled and split


# ------------------------------------------------------------------------------------------------ GPU
def host_batches(model, structs, flags, batch_size, table=None):
    """``predict(..., local_attention=True)`` on the padded ``DataIterator(..., use_ring=True)`` batches of the same
    structures in the shape classes of ``predict_structures``: per structure (y, ga [n], la [L, H, P_s])."""
    from scann_b200 import voronoi as V
    from scann_b200.datagenerator import DataIterator, pack_padded
    from scann_b200.model import shape_class
    de, dn = ring_rows(structs, V.compute_voronoi_neighbors(structs), flags)
    kw = dict(feature="cgcnn", atomic_features=table) if table is not None else {}
    it = DataIterator(de, dn, batch_size=batch_size, g_update=bool(model.spec.g_update), use_ring=True, **kw)
    out = []
    for i in range(len(it)):
        csr, _ = it.csr_item(i)
        csr = dict(csr)
        csr["M"], csr["N"] = shape_class(csr["M"], csr["N"])
        inputs = pack_padded(csr)                          # DataIterator.__getitem__ on the shape class
        if table is not None:
            inputs["atomic"] = table[inputs["atomic"]]
        y, ga, la = model.predict(inputs, local_attention=True)
        sa, an = csr["struct_atom_off"], csr["atom_nbr_off"]
        for s in range(len(sa) - 1):
            n = sa[s + 1] - sa[s]
            cols = [la[:, s, :, m, :an[sa[s] + m + 1] - an[sa[s] + m]] for m in range(n)]
            out.append((y[s, 0], ga[s, :n, 0], np.concatenate(cols, axis=2)))
    return out


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _ptgp_case():
    structs, flags = ptgp_like(10, seed=72)              # batches of M = 256, 256 and 184 (shape classes)
    return structs, flags, 4


def _qm9_case():
    structs = qm9_like(30, seed=12)
    structs[9:9] = [hub()]                                 # one batch with > 32 neighbours: the 64-row plan
    return structs, random_flags(structs, seed=2), 16


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["ptgp", "qm9", "cgcnn"])
def test_predict_structures_equals_the_padded_ring_batches(case):
    """y, ga and every layer's local-attention scores bit for bit, in the same shape classes."""
    from scann_b200.synth import cgcnn_table
    table = None
    if case == "ptgp":
        model, _ = _ring_model("ptgp", **PTGP)              # the shipped 11 layers
        structs, flags, bs = _ptgp_case()
    else:
        feature = "cgcnn" if case == "cgcnn" else "atomic"
        model, _ = _ring_model("qm9", n_attention=2, feature=feature)
        structs, flags, bs = _qm9_case()
        if case == "cgcnn":
            table = cgcnn_table()
            table[0] = 0.25
    y, ga, la = model.predict_structures(structs, batch_size=bs, local_attention=True, atomic_features=table,
                                         ring_aromatic=flags)
    want = host_batches(model, structs, flags, bs, table)
    assert len(want) == len(structs) == len(ga) == len(la)
    for k, (y_h, ga_h, la_h) in enumerate(want):
        assert _bits(y[k, 0]) == _bits(y_h), k
        assert np.array_equal(_bits(ga[k]), _bits(ga_h)), k
        assert np.array_equal(_bits(la[k].scores), _bits(la_h)), k
    Ms = [b.M for b in model.engine._batches.values()]
    if case == "ptgp":
        assert max(Ms) > 193 and min(Ms) <= 193, Ms        # above and within the staged GlobalAttention capacity
    else:
        assert any(b.N > 32 for b in model.engine._batches.values())
    model.engine.check_status()


@pytest.mark.gpu
def test_the_flags_of_one_structure_change_its_output_only():
    model, _ = _ring_model("ptgp", **PTGP)
    structs, flags, bs = _ptgp_case()
    y0, ga0 = model.predict_structures(structs, batch_size=bs, ring_aromatic=flags)
    changed = [f.copy() for f in flags]
    k = 5                                                  # the second structure of the second batch
    changed[k] = 1 - changed[k]
    y1, ga1 = model.predict_structures(structs, batch_size=bs, ring_aromatic=changed)
    y2, _ = model.predict_structures(structs, batch_size=bs, ring_aromatic=flags)
    assert _bits(y1[k, 0]) != _bits(y0[k, 0]) and not np.array_equal(ga1[k], ga0[k])
    others = [i for i in range(len(structs)) if i != k]
    assert np.array_equal(_bits(y1[others]), _bits(y0[others]))
    assert all(np.array_equal(ga1[i], ga0[i]) for i in others)
    assert np.array_equal(_bits(y2), _bits(y0))            # and back: no flag of the last call stays behind


@pytest.mark.gpu
def test_a_ptgp_batch_against_the_fp64_oracle():
    import torch
    from oracle import scann_oracle as O
    from scann_b200 import voronoi as V
    from scann_b200.datagenerator import prepare_input_from_neighbors
    from scann_b200.params import ParamLayout
    from tests.golden.make_golden import oracle_kwargs
    from tests.test_gpu_parity import TOL_OUT, rel
    model, _ = _ring_model("ptgp", **PTGP)
    spec = model.spec
    structs, flags, bs = _ptgp_case()
    structs, flags = structs[:bs], flags[:bs]             # one batch
    y, ga = model.predict_structures(structs, batch_size=bs, ring_aromatic=flags)
    wd = ParamLayout(spec).to_dict(model.engine.get_params())
    lists = V.compute_voronoi_neighbors(structs)
    for k, s in enumerate(structs):
        inp = prepare_input_from_neighbors(list(s.atomic_numbers), lists[k], angle=bool(spec.g_update))
        inp["ring_aromatic"] = np.asarray(flags[k], np.int32)[None]
        y_ref, ga_ref = O.predict(wd, inp, use_ring=True, **oracle_kwargs(spec))
        # a single output of a cancelling sum: bounded by TOL_OUT or 5 x the distance of the reference's own fp32
        # arithmetic (fp32 oracle) from fp64, as in tests/test_cgcnn_routes.py
        y32, _ = O.predict(wd, inp, torch.float32, use_ring=True, **oracle_kwargs(spec))
        tol_y = max(TOL_OUT, 5.0 * rel(np.ravel(y32), np.ravel(y_ref)))
        assert rel(y[k], np.ravel(y_ref)) <= tol_y and rel(ga[k], np.ravel(ga_ref)) <= TOL_OUT, k


def _buffers(b):
    return {k: getattr(b, k).clone() for k in ("atomic", "atom_mask", "nbr", "nmask", "weight", "dist", "target",
                                               "ring")}


@pytest.mark.gpu
@pytest.mark.parametrize("angle", [True, False])
def test_from_structures_buffers_equal_the_host_route_for_three_shuffled_epochs(monkeypatch, angle):
    import torch
    from scann_b200 import model as Mo
    from scann_b200 import voronoi as V
    from scann_b200.datagenerator import DataIterator, DeviceDataIterator
    p_structs, p_flags = ptgp_like(6, seed=3)
    q_structs = qm9_like(40, seed=13)
    structs, flags = p_structs + q_structs, p_flags + random_flags(q_structs, seed=4)
    y = np.random.default_rng(0).standard_normal(len(structs)).tolist()
    monkeypatch.setattr(Mo, "_CHUNK_ATOMS", 600)           # several chunks: their CSR is joined on the device
    de, dn = ring_rows(structs, V.compute_voronoi_neighbors(structs), flags, y)
    np.random.seed(9)
    host = DataIterator(de, dn, batch_size=8, shuffle=True, use_ring=True, converter=True, g_update=angle)
    np.random.seed(9)
    dev = DeviceDataIterator.from_structures(structs, y, batch_size=8, shuffle=True, g_update=angle, use_ring=True,
                                             ring_aromatic=flags, converter=True)
    assert dev.use_ring and dev.ring.dtype == torch.int32 and tuple(dev.ring.shape) == (len(host.ring), 2)
    eng = _ring_model("ptgp", n_attention=1, infer=False, **PTGP)[0].engine      # embeds C, Pt and H..F
    for ep in range(3):
        assert np.array_equal(host.indexes, dev.indexes)
        for i in range(len(host)):
            want = _buffers(eng.load_batch_csr(*host.csr_item(i), plan=False))
            got = _buffers(eng.load_batch_gather(dev, *dev.batch_shape(i), plan=False))
            for k in want:
                assert torch.equal(got[k].view(torch.uint8), want[k].view(torch.uint8)), (ep, i, k)
        np.random.seed(100 + ep)
        host.on_epoch_end()
        np.random.seed(100 + ep)
        dev.on_epoch_end()
    (ih, _), (id_, _) = host[0], dev[0]
    assert np.array_equal(ih["ring_aromatic"], id_["ring_aromatic"])
    eng.check_status()


def _fit(route, cfg_name, over, structs, flags, y, n_train, bs):
    from scann_b200 import voronoi as V
    from scann_b200.datagenerator import DataIterator, DeviceDataIterator
    g = bool(over.get("g_update", True))
    if route == "host":
        de, dn = ring_rows(structs, V.compute_voronoi_neighbors(structs), flags, y)
        np.random.seed(21)
        it = DataIterator(de[:n_train], dn[:n_train], batch_size=bs, shuffle=True, g_update=g, use_ring=True)
        vit = DataIterator(de[n_train:], dn[n_train:], batch_size=bs, g_update=g, use_ring=True)
    else:
        np.random.seed(21)
        it = DeviceDataIterator.from_structures(structs[:n_train], y[:n_train], batch_size=bs, shuffle=True, g_update=g,
                                                use_ring=True, ring_aromatic=flags[:n_train])
        vit = DeviceDataIterator.from_structures(structs[n_train:], y[n_train:], batch_size=bs, g_update=g,
                                                 use_ring=True, ring_aromatic=flags[n_train:])
    m, _ = _ring_model(cfg_name, seed=4, infer=False, deterministic=True, **over)
    m.compile(optimizer=5e-4)
    hist = m.fit(it, epochs=2, validation_data=vit, verbose=0)
    eng = m.engine
    assert eng.train_dropout and eng.deterministic
    return {"hist": hist.history, "params": eng.params.cpu().numpy(), "m": eng.adam_m.cpu().numpy(),
            "v": eng.adam_v.cpu().numpy(), "rng": np.random.get_state()}


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["ptgp", "qm9"])
def test_deterministic_fit_gives_the_same_bits_on_both_routes(case):
    if case == "ptgp":
        structs, flags = ptgp_like(24, seed=5)
        cfg_name, over, n_train, bs = "ptgp", dict(PTGP, n_attention=3), 16, 8
    else:
        structs = qm9_like(160, seed=6)
        flags = random_flags(structs, seed=7)
        cfg_name, over, n_train, bs = "qm9", {"n_attention": 2}, 128, 32
    y = np.random.default_rng(1).standard_normal(len(structs)).tolist()
    h = _fit("host", cfg_name, over, structs, flags, y, n_train, bs)
    d = _fit("device", cfg_name, over, structs, flags, y, n_train, bs)
    assert h["hist"] == d["hist"] and len(d["hist"]["val_mae"]) == 2
    for k in ("params", "m", "v"):
        assert np.array_equal(h[k].view(np.uint32), d[k].view(np.uint32)), k
    st_h, st_d = h["rng"], d["rng"]
    assert st_h[0] == st_d[0] and np.array_equal(st_h[1], st_d[1]) and st_h[2:] == st_d[2:]


@pytest.mark.gpu
def test_prepare_structures_trains_and_evaluates_like_prepare_dataset(tmp_path, monkeypatch):
    from scann_b200 import voronoi as V
    from scann_b200.configs import get_config
    from scann.models import SCANN
    monkeypatch.setenv("TF_DETERMINISTIC_OPS", "1")
    structs = qm9_like(80, seed=12)
    flags = random_flags(structs, seed=8)
    y = np.random.default_rng(3).standard_normal(len(structs)).tolist()
    recs = np.empty(len(structs), object)
    for k, (s, t) in enumerate(zip(structs, y)):
        recs[k] = {"Atomic": list(s.atomic_numbers), "Properties": {"homo": t},
                   "Features": {"ring": flags[k][:, 0], "aromatic": flags[k][:, 1]}}
    nbrs = np.empty(len(structs), object)
    for k, lists in enumerate(V.compute_voronoi_neighbors(structs)):
        nbrs[k] = lists
    np.save(tmp_path / "data.npy", recs, allow_pickle=True)
    np.save(tmp_path / "nbr.npy", nbrs, allow_pickle=True)

    def run(name, prepare):
        cfg = get_config("qm9")
        cfg["model"].update(n_attention=2, use_ring=True)
        cfg["hyper"].update(batch_size=16, test_percent=0.1, train_size=None, test_size=None,
                            save_path=str(tmp_path / name), data_energy_path=str(tmp_path / "data.npy"),
                            data_nei_path=str(tmp_path / "nbr.npy"))
        np.random.seed(7)
        s = SCANN(cfg, mode="train")
        prepare(s)
        s.train(2)
        s.evaluate()
        run_dir = str(tmp_path / f"{name}_homo")
        with open(os.path.join(run_dir, "report.txt")) as f:
            report = f.read()
        return report, np.load(os.path.join(run_dir, "hist_data.npy"), allow_pickle=True), s

    rep_h, hist_h, sh = run("host", lambda s: s.prepare_dataset())
    rep_d, hist_d, sd = run("device", lambda s: s.prepare_structures(structs, y, ring_aromatic=flags))
    assert sh.config["hyper"]["target_mean"] == sd.config["hyper"]["target_mean"]
    assert sh.config["hyper"]["data_size"] == sd.config["hyper"]["data_size"] == len(structs)
    assert type(sd.testIter).__name__ == "DeviceDataIterator" and sd.testIter.use_ring
    assert sh.trainIter.use_ring and np.array_equal(sh.testIter.ring, sd.testIter.ring.cpu().numpy())
    assert rep_h == rep_d
    assert list(hist_h[0]) == list(hist_d[0]) and list(hist_h[1]) == list(hist_d[1]) and hist_h[2] == hist_d[2]
