"""Pins against REFERENCE-RUN code: the reference's own ``DataIterator.__getitem__``
(scann/utils/datagenerator.py:69-135), ``pad_sequence`` / ``pad_nested_sequences`` (scann/utils/general.py:14-50),
``SGDRC`` (scann/layers/custom_layers.py:78-179) and ``configs/*.yaml`` are imported from the reference checkout
named by SCANN_REFERENCE_ROOT (tests/ref_stubs.py replaces TensorFlow / pymatgen / openbabel / ase by inert stubs; the
code under test is plain numpy / Python) and compared bit for bit with this repo's implementations and with the
oracle restatement.

The values these comparisons found are stored in ``tests/golden/reference/pins_*.npz`` (tests/ref_stubs.check_stored):
every test checks this repo's implementation against them, and, where the reference checkout is present, also against
the reference live.  They were recorded from this repo's implementations as last compared equal with the reference.
The floating-point layers (attention.py) are pinned by tests/test_reference_graph.py and the oracle."""
import warnings

import numpy as np
import pytest

from tests import ref_stubs
from tests.ref_stubs import check_stored


@pytest.fixture(scope="module")
def ref():
    """The reference's own objects, or None where its source is absent (the stored values stand in)."""
    if not ref_stubs.reference_available():
        return None
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return ref_stubs.load_reference()


def _digest(a):
    """SHA-256 of an array's dtype, shape and bytes: a bit-for-bit comparison that stores 64 characters."""
    import hashlib
    a = np.ascontiguousarray(a)
    return np.array(hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest())


def _batches(it):
    """Every batch of an iterator as flat name -> digest."""
    out = {"len": np.int64(len(it))}
    for i in range(len(it)):
        inputs, target = it[i]
        out[f"b{i}/target"] = _digest(target)
        for k, v in inputs.items():
            out[f"b{i}/{k}"] = _digest(v)
    return out


@pytest.mark.skipif(not ref_stubs.reference_available(), reason=ref_stubs.SKIP_REASON)
def test_the_objects_are_the_references_own(ref):
    import os
    root = os.path.realpath(ref_stubs.REFERENCE_ROOT)
    for mod in ("datagenerator", "general", "custom_layers"):
        assert os.path.realpath(ref[mod].__file__).startswith(root)
    assert ref["DataIterator"].__module__ == "scann.utils.datagenerator"
    assert "tensorflow" in ref["stubbed"]                      # the import really went through the stubs
    import scann                                               # and this repo's alias package is back in place
    assert not os.path.realpath(scann.__file__).startswith(root)


@pytest.mark.parametrize("g_update,use_ring,converter", [(True, False, False), (False, True, False), (False, False, True)])
def test_dataiterator_matches_the_reference_class_bit_for_bit(ref, g_update, use_ring, converter):
    """Every batch of a ragged synthetic data set, incl. the last partial one and a 1000-padded neighbour slot."""
    from oracle import datagen_oracle as DO
    from scann_b200.datagenerator import DataIterator, synthetic_ragged
    de, dn = synthetic_ragged(53, seed=7, use_ring=use_ring)
    dn[0][0][0] = (0, 1000, 0.0, 0.0, 0.0)                     # the reference's own padding marker inside a list
    ours = DataIterator(de, dn, batch_size=8, converter=converter, use_ring=use_ring, g_update=g_update)
    assert len(ours) == 7
    check_stored(f"pins_dataiterator_{int(g_update)}{int(use_ring)}{int(converter)}",
                 dict(_batches(ours), weight_index=np.int64(ours.weight_index)))
    for i in range(len(ours)):
        o_in, o_e = ours[i]
        idx = list(range(i * 8, min(53, (i + 1) * 8)))
        p_in, p_e = DO.get_item(de, dn, idx, g_update=g_update, use_ring=use_ring, converter=1000 if converter else 1.0)
        assert np.array_equal(p_e, o_e) and p_e.dtype == o_e.dtype and set(p_in) == set(o_in)
        for k in o_in:
            assert p_in[k].dtype == o_in[k].dtype and np.array_equal(p_in[k], o_in[k]), ("oracle.datagen_oracle", k)
    if ref is None:
        return
    theirs = ref["DataIterator"](de, dn, batch_size=8, converter=converter, use_ring=use_ring, g_update=g_update)
    assert len(theirs) == len(ours)
    assert theirs.weight_index == ours.weight_index
    for i in range(len(theirs)):
        r_in, r_e = theirs[i]
        o_in, o_e = ours[i]
        assert np.array_equal(o_e, r_e) and o_e.dtype == r_e.dtype
        assert set(o_in) == set(r_in)
        for k in r_in:
            assert o_in[k].dtype == r_in[k].dtype and o_in[k].shape == r_in[k].shape, k
            assert np.array_equal(o_in[k], r_in[k]), k


def test_dataiterator_shuffle_follows_numpy_global_rng_like_the_reference(ref):
    from scann_b200.datagenerator import DataIterator, synthetic_ragged
    de, dn = synthetic_ragged(20, seed=2)
    np.random.seed(123)
    ours = DataIterator(de, dn, batch_size=6, shuffle=True)
    check_stored("pins_dataiterator_shuffle", dict(_batches(ours), indexes=np.asarray(ours.indexes)))
    if ref is None:
        return
    np.random.seed(123)
    theirs = ref["DataIterator"](de, dn, batch_size=6, shuffle=True)
    assert np.array_equal(theirs.indexes, ours.indexes)
    for i in range(len(theirs)):
        assert np.array_equal(theirs[i][1], ours[i][1])
        assert np.array_equal(theirs[i][0]["neighbors"], ours[i][0]["neighbors"])


def test_pad_helpers_match_the_reference(ref):
    """prepare_input_from_neighbors (the padding half of general.py:206-246) against the reference's pad_sequence."""
    from oracle import datagen_oracle as DO
    from scann_b200.datagenerator import prepare_input_from_neighbors
    rng = np.random.default_rng(0)
    na = 11
    neighbors = [[(0, int(rng.integers(0, na)), float(rng.uniform(0.4, 3)), float(rng.uniform(0.2, 1)), float(rng.uniform(1, 4)))
                  for _ in range(int(rng.integers(1, 9)))] for _ in range(na)]
    z = rng.choice([1, 6, 7, 8], size=na).astype(np.int32)
    stored = {}
    for angle in (True, False):
        got = prepare_input_from_neighbors(z, neighbors, angle=angle)
        stored.update({f"{angle}/{k}": v for k, v in got.items()})
        assert np.array_equal(got["atomic"], np.array([z], "int32"))
        assert np.array_equal(got["atom_mask"], np.expand_dims(np.array([z]) != 0, -1))
        if ref is None:
            continue
        pad = ref["pad_sequence"]
        local = np.array([pad([[n[1] for n in lc] for lc in neighbors], value=1000)], "int32")
        mask = local != 1000
        local[local == 1000] = 0
        w = np.array([pad([[n[2 if angle else 3] for n in lc] for lc in neighbors], dtype="float32")])
        d = np.array([pad([[n[-1] for n in lc] for lc in neighbors], dtype="float32")])
        assert np.array_equal(got["neighbors"], local) and got["neighbors"].dtype == local.dtype
        assert np.array_equal(got["neighbor_mask"], mask)
        assert np.array_equal(got["neighbor_weight"], w) and got["neighbor_weight"].dtype == w.dtype
        assert np.array_equal(got["neighbor_distance"], d)
    # pad_nested_sequences: the 3-D padding of DataIterator
    nested = [[[1, 2], [3]], [[4, 5, 6]]]
    stored["nested"] = DO.pad_nested_sequences(nested, 3, 2, "int32", value=1000)
    check_stored("pins_pad_helpers", stored)
    if ref is not None:
        assert np.array_equal(stored["nested"], ref["pad_nested_sequences"](nested, 3, 2, value=1000, dtype="int32"))


SGDRC_CASES = [dict(lr_max=5e-4, lr_min=1e-4, t0=50, tmult=2, lr_max_compression=1.2, trigger_val_mae=80),
               dict(lr_max=1e-3, lr_min=1e-5, t0=10, tmult=1, lr_max_compression=5, trigger_val_mae=9999),
               dict(lr_max=1e-3, lr_min=1e-5, t0=7, tmult=3, lr_max_compression=0, trigger_val_mae=0.5)]
SGDRC_ATTRS = ("triggered", "lr_warmup_next", "lr_warmup_current", "lr", "ti", "tcur", "best_val_mae")


@pytest.mark.parametrize("kw", SGDRC_CASES)
def test_sgdrc_matches_the_reference_over_a_200_epoch_trace(ref, kw):
    """The warm-restart schedule, driven exactly as keras drives it: LearningRateScheduler calls lr_scheduler(epoch) at
    the start of an epoch, the callback's on_epoch_end(epoch, logs) closes it."""
    from scann_b200.callbacks import SGDRC
    schedulers = [SGDRC(show_lr=False, **kw)] + ([ref["SGDRC"](show_lr=False, **kw)] if ref is not None else [])
    rng = np.random.default_rng(5)
    val = 100.0 * np.exp(-np.arange(200) / 60.0) * (1.0 + 0.2 * rng.standard_normal(200)) + 0.3
    for s in schedulers:
        s.on_train_begin({})
    lrs, attrs = np.zeros(200), np.zeros((200, len(SGDRC_ATTRS)))
    for ep in range(200):
        a = [s.lr_scheduler(ep) for s in schedulers]
        assert all(x == a[0] for x in a), (ep, a)               # bit-identical floats
        lrs[ep] = a[0]
        for s in schedulers:
            s.on_epoch_end(ep, {"val_mae": float(val[ep])})
        for j, attr in enumerate(SGDRC_ATTRS):
            v = [getattr(s, attr) for s in schedulers]
            assert all(x == v[0] for x in v), (ep, attr)
            attrs[ep, j] = v[0]
    check_stored(f"pins_sgdrc_{SGDRC_CASES.index(kw)}", {"lr": lrs, "attrs": attrs})
    assert schedulers[0].triggered == (val.min() <= kw["trigger_val_mae"])


def test_shipped_yaml_configs_equal_the_restated_dicts():
    """configs/*.yaml of the reference through load_yaml == scann_b200/configs.py (the keys the hot path reads)."""
    import json
    import os
    from scann_b200.config import load_yaml
    from scann_b200.configs import CONFIGS
    # the restated dicts as last found equal to the shipped files
    check_stored("pins_configs", {"json": np.array(json.dumps(CONFIGS, sort_keys=True))})
    if not ref_stubs.reference_available():
        return
    cdir = os.path.join(ref_stubs.REFERENCE_ROOT, "configs")
    shipped = sorted(f[len("model_"):-len(".yaml")] for f in os.listdir(cdir) if f.startswith("model_") and f.endswith(".yaml"))
    assert shipped == sorted(CONFIGS), (shipped, sorted(CONFIGS))           # every yaml the reference ships is restated
    for name, mine in CONFIGS.items():
        theirs = load_yaml(os.path.join(cdir, f"model_{name}.yaml"))
        for section in ("model", "hyper"):
            for k, v in mine[section].items():
                assert k in theirs[section], (name, section, k)
                assert theirs[section][k] == v, (name, section, k, theirs[section][k], v)
        # nothing the graph builder reads is missing from the restatement (scann_model.py:330-434)
        for k in ("n_atoms", "embedding_dim", "local_dim", "num_head", "use_attn_norm", "n_attention", "global_dim",
                  "use_ga_norm", "dense_out", "use_ring"):
            assert theirs["model"][k] == mine["model"][k], (name, k)
        assert ("g_update" in theirs["model"]) == ("g_update" in mine["model"]), name     # model_ptgp.yaml lacks it


@pytest.mark.skipif(not ref_stubs.reference_available(), reason=ref_stubs.SKIP_REASON)
def test_cgcnn_dataiterator_matches_the_reference_class(ref):
    """feature='cgcnn' (datagenerator.py:107-110): the atom mask comes from the atomic numbers, then the numbers are
    replaced by the 92-vectors of the reference's own ``atomic_features`` table (handed over at run time: the table is
    data of the CGCNN project and is not shipped here, so this comparison cannot run without the reference)."""
    from scann_b200.datagenerator import DataIterator, synthetic_ragged
    de, dn = synthetic_ragged(21, seed=3)
    theirs = ref["DataIterator"](de, dn, batch_size=8, feature="cgcnn", g_update=True)
    ours = DataIterator(de, dn, batch_size=8, feature="cgcnn", g_update=True, atomic_features=ref["atomic_features"])
    for i in range(len(theirs)):
        (r_in, r_e), (o_in, o_e) = theirs[i], ours[i]
        assert np.array_equal(r_e, o_e) and set(r_in) == set(o_in)
        assert o_in["atomic"].shape[-1] == 92
        for k in r_in:
            assert o_in[k].dtype == r_in[k].dtype and np.array_equal(o_in[k], r_in[k]), k
    assert not hasattr(ours, "feature") or ours.feature == "cgcnn"


SPLIT_CASES = [dict(len_data=1000), dict(len_data=1003, test_percent=0.15),
               dict(len_data=500, train_size=400, test_size=60), dict(len_data=17, test_percent=0.2)]


@pytest.mark.parametrize("kw", SPLIT_CASES)
def test_split_data_matches_the_reference_function(ref, kw):
    from scann_b200.datagenerator import split_data
    np.random.seed(11)
    ours = split_data(**kw)
    assert len(ours) == 4
    check_stored(f"pins_split_data_{SPLIT_CASES.index(kw)}", {str(j): a for j, a in enumerate(ours)})
    if ref is None:
        return
    np.random.seed(11)
    theirs = ref["general"].split_data(**kw)
    assert len(theirs) == 4
    for a, b in zip(theirs, ours):
        assert a.dtype == b.dtype and np.array_equal(a, b)


def _write_dataset(tmp_path, n=37, ring=True, seed=5):
    """A data set in the format the reference's preprocessing writes (scann/utils/dataset/qm9.py): records with
    Atomic / Properties / Features, and the per-structure neighbour lists."""
    from scann_b200.datagenerator import synthetic_ragged
    rng = np.random.default_rng(seed)
    de, dn = synthetic_ragged(n, seed=seed, use_ring=True)
    records = []
    for z, _, flags in de:
        flags = np.asarray(flags)
        records.append({"Atomic": list(z), "Properties": {"homo": float(rng.normal(-6.5, 0.6)), "u0": float(rng.normal(-400, 40)),
                                                          "Ref_energy": float(rng.normal(-399, 40))},
                        "Features": {"Ring": flags[:, 0], "Aromatic": flags[:, 1]}})
    p_e, p_n = str(tmp_path / "data_energy.npy"), str(tmp_path / "data_neighbor.npy")
    np.save(p_e, np.array(records, dtype=object), allow_pickle=True)
    np.save(p_n, np.array(dn, dtype=object), allow_pickle=True)
    return p_e, p_n


LOAD_CASES = [(False, True, "homo"), (True, False, "u0"), (False, False, "homo"), (True, True, "u0")]


@pytest.mark.parametrize("use_ref,use_ring,target", LOAD_CASES)
def test_load_dataset_matches_the_reference_function(ref, tmp_path, use_ref, use_ring, target):
    from scann_b200.datagenerator import load_dataset
    p_e, p_n = _write_dataset(tmp_path)
    oe, on = load_dataset(p_e, p_n, target, use_ref=use_ref, use_ring=use_ring)
    assert oe.dtype == object
    stored = {"shape": np.array(oe.shape), "target": np.array([r[1] for r in oe], np.float64),
              "atomic_len": np.array([len(r[0]) for r in oe]), "atomic": np.concatenate([np.asarray(r[0]) for r in oe]),
              "pairs_len": np.array([len(lc) for nb in on for lc in nb]),
              "pairs": _digest(np.array([pair for nb in on for lc in nb for pair in lc], np.float64))}
    if use_ring:
        stored["ring"] = np.concatenate([np.asarray(r[2]) for r in oe])
    check_stored(f"pins_load_dataset_{LOAD_CASES.index((use_ref, use_ring, target))}", stored)
    if ref is None:
        return
    te, tn = ref["general"].load_dataset(p_e, p_n, target, use_ref=use_ref, use_ring=use_ring)
    assert te.shape == oe.shape and te.dtype == oe.dtype == object and tn.shape == on.shape
    for a, b in zip(te, oe):
        assert list(a[0]) == list(b[0]) and a[1] == b[1]
        if use_ring:
            assert np.array_equal(a[2], b[2])
    for a, b in zip(tn, on):
        assert a == b


def test_pad_helpers_of_the_package_match_the_reference_functions(ref):
    from scann.utils import pad_nested_sequences, pad_sequence          # the reference's import path, this repo's code
    from scann_b200 import datagenerator as dg
    assert pad_sequence is dg.pad_sequence
    rng = np.random.default_rng(9)
    seqs = [list(rng.integers(1, 50, size=int(n))) for n in rng.integers(1, 12, size=9)]
    calls = [(pad_sequence, ref and ref["pad_sequence"], seqs, kw)
             for kw in (dict(), dict(maxlen=15, value=1000), dict(maxlen=4), dict(dtype="float32", value=-1.5))]
    feats = [rng.integers(0, 2, size=(int(n), 2)) for n in rng.integers(1, 8, size=5)]      # ring flags: [atoms, 2]
    calls.append((pad_sequence, ref and ref["pad_sequence"], feats, dict(maxlen=9)))
    nested = [[list(rng.random(int(k))) for k in rng.integers(0, 7, size=int(n))] for n in rng.integers(1, 6, size=7)]
    calls += [(pad_nested_sequences, ref and ref["pad_nested_sequences"], nested, kw)
              for kw in (dict(max_len_1=7, max_len_2=6, dtype="float32"),
                         dict(max_len_1=9, max_len_2=8, dtype="float32", value=3.0),
                         dict(max_len_1=3, max_len_2=2, dtype="float32"))]
    stored = {}
    for j, (ours, theirs, data, kw) in enumerate(calls):
        stored[str(j)] = b = ours(data, **kw)
        if theirs is not None:
            a = theirs(data, **kw)
            assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b), kw
    assert stored["4"].shape == (5, 9, 2)
    check_stored("pins_pad_helpers_package", stored)


def test_prepare_input_pmt_matches_the_reference_function(ref, monkeypatch):
    """The reference's OWN ``prepare_input_pmt`` (general.py:206-246) with its Voronoi search replaced by given
    neighbour lists, beside ``scann.utils.prepare_input_pmt(struct, ..., neighbors=...)``: identical input dicts
    (README.md:102-120 inference flow); without neighbours ours refuses loudly."""
    import types
    from scann.utils import prepare_input_pmt
    rng = np.random.default_rng(4)
    na = 14
    neighbors = [[(0, int(rng.integers(0, na)), float(rng.uniform(0.4, 3)), float(rng.uniform(0.2, 1)), float(rng.uniform(1, 4)))
                  for _ in range(int(rng.integers(1, 12)))] for _ in range(na)]
    struct = types.SimpleNamespace(atomic_numbers=tuple(int(z) for z in rng.choice([1, 6, 7, 8, 26], size=na)))
    seen = {}
    if ref is not None:
        monkeypatch.setattr(ref["general"], "compute_voronoi_neighbor",
                            lambda s, d_thresh, w_thresh: (seen.update(d=d_thresh, w=w_thresh), neighbors)[1])
    stored = {}
    for angle in (True, False):
        got = prepare_input_pmt(struct, d_t=3.5, w_t=0.3, angle=angle, neighbors=neighbors)
        stored.update({f"{angle}/{k}": v for k, v in got.items()})
        if ref is None:
            continue
        want = ref["general"].prepare_input_pmt(struct, d_t=3.5, w_t=0.3, angle=angle)
        assert seen == {"d": 3.5, "w": 0.3}
        assert set(got) == set(want)
        for k in want:
            assert got[k].dtype == want[k].dtype and got[k].shape == want[k].shape and np.array_equal(got[k], want[k]), k
    check_stored("pins_prepare_input_pmt", stored)
    with pytest.raises(NotImplementedError):
        prepare_input_pmt(struct)
