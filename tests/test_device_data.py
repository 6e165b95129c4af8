"""Training from a device-resident data set: ``DeviceDataIterator`` + ``Engine.load_batch_gather``
(``scann_gather_batch``, csrc/plan.cu).

The host route it replaces is ``DataIterator.csr_item`` -> ``Engine.load_batch_csr`` every step; the device route must
give the same padded buffers, the same shape classes and, in the deterministic mode, the same training bits."""
import os
import types

import numpy as np
import pytest

from tests.test_predict_structures import qm9_like
from tests.test_voronoi import _gpu_cases, struct

NOUP_RING = {"g_update": False, "gaussian_d": 4.0, "use_ring": True}


def ragged_set(n, seed=0, use_ring=False, max_atoms=20, max_nbr=12):
    """synthetic_ragged with the reference's padding marker 1000 in some lists and an atom without neighbours."""
    from scann_b200.datagenerator import synthetic_ragged
    de, dn = synthetic_ragged(n, seed=seed, max_atoms=max_atoms, max_nbr=max_nbr, use_ring=use_ring)
    rng = np.random.default_rng(seed + 1)
    for s in rng.choice(n, n // 5, replace=False):
        lists = dn[s]
        a = int(rng.integers(len(lists)))
        lists[a] = [(0, 1000, 0.5, 0.5, 2.0) if k % 2 else t for k, t in enumerate(lists[a])]
    dn[1][0] = []
    return de, dn


def host_only(it):
    """A DeviceDataIterator with the host arrays of ``it`` and no device arrays (enough for the epoch order and the
    batch shapes)."""
    from scann_b200.datagenerator import DeviceDataIterator
    pair_off, nmax, npairs = DeviceDataIterator.host_sizes(it.atom_off, it.nbr_off, it.nbr_idx)
    return DeviceDataIterator({}, it.energy, it.atom_off, pair_off, nmax, npairs, batch_size=it.batch_size,
                              shuffle=it.shuffle, weight_index=it.weight_index, converter=it.converter)


# ------------------------------------------------------------------------------------------------ CPU
def test_gather_batch_is_declared_exported_and_bound():
    from scann_b200 import _abi
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                            "scann_b200.h")).read()
    assert "int scann_gather_batch(" in hdr and "scann_gather_batch" in _abi.PROTOTYPES
    assert hasattr(_abi.lib, "scann_gather_batch")


def test_shuffle_consumes_the_global_generator_like_data_iterator():
    from scann_b200.datagenerator import DataIterator
    de, dn = ragged_set(77)
    np.random.seed(11)
    host = DataIterator(de, dn, batch_size=16, shuffle=True)
    orders_h = [host.indexes.copy()]
    for _ in range(3):
        host.on_epoch_end()
        orders_h.append(host.indexes.copy())
    state_h = np.random.get_state()
    np.random.seed(11)
    dev = host_only(DataIterator(de, dn, batch_size=16, shuffle=False))
    dev.shuffle = True
    dev.on_epoch_end()
    orders_d = [dev.indexes.copy()]
    for _ in range(3):
        dev.on_epoch_end()
        orders_d.append(dev.indexes.copy())
    state_d = np.random.get_state()
    assert all(np.array_equal(a, b) for a, b in zip(orders_h, orders_d))
    assert state_h[0] == state_d[0] and np.array_equal(state_h[1], state_d[1]) and state_h[2:] == state_d[2:]
    assert len(dev) == len(host) == 5


def test_batch_shapes_are_those_of_csr_item():
    from scann_b200.datagenerator import DataIterator
    de, dn = ragged_set(77)
    np.random.seed(2)
    host = DataIterator(de, dn, batch_size=16, shuffle=True)
    dev = host_only(host)
    dev.indexes = host.indexes.copy()
    for i in range(len(host)):
        csr, e = host.csr_item(i)
        start, B, M, N, P = dev.batch_shape(i)
        assert (start, B, M, N, P) == (16 * i, len(e), csr["M"], csr["N"], int(np.count_nonzero(csr["nbr_idx"] != 1000)))
        assert np.array_equal(dev.batch_target(i), e)
    assert dev.nmax[1] >= 1 and (host.nbr_idx == 1000).any()


def test_refusals_name_the_reason_and_the_structure():
    from scann_b200.datagenerator import DeviceDataIterator as D
    with pytest.raises(NotImplementedError, match="cgcnn"):
        D.from_data_iterator(types.SimpleNamespace(feature="cgcnn"))
    with pytest.raises(NotImplementedError, match="cgcnn"):
        D.from_structures([], [], feature="cgcnn")
    with pytest.raises(NotImplementedError, match="use_ring.*openbabel"):
        D.from_structures([], [], use_ring=True)
    ok = struct(np.eye(3) * 5.0, [[0.0, 0.0, 0.0]], [6])
    empty = types.SimpleNamespace(lattice=types.SimpleNamespace(matrix=np.eye(3) * 5.0), cart_coords=np.zeros((0, 3)),
                                  atomic_numbers=[])
    with pytest.raises(ValueError, match="structure 1 has no sites"):
        D.from_structures([ok, empty], [0.0, 1.0])
    rng = np.random.default_rng(0)
    big = struct(np.eye(3) * 60.0, rng.uniform(0, 60, (1001, 3)), [6] * 1001)
    with pytest.raises(ValueError, match="structure 2 has 1001 sites: at most 1000"):
        D.from_structures([ok, ok, big], [0.0, 1.0, 2.0])
    with pytest.raises(ValueError, match="3 structures but 2 targets"):
        D.from_structures([ok, ok, ok], [0.0, 1.0])
    # a data set with 2^31 pairs: the int32 offsets are refused before anything is uploaded
    huge = types.SimpleNamespace(feature="atomic", atom_off=np.array([0, 1, 2, 3]),
                                 nbr_off=np.array([0, 2 ** 30, 2 ** 31 - 1, 2 ** 31 + 5]))
    with pytest.raises(ValueError, match="structure 2: the data set's neighbour pairs exceed int32"):
        D.from_data_iterator(huge)


# ------------------------------------------------------------------------------------------------ GPU
def _model(over=None, n_attention=2, seed=4, cfg_name="qm9", deterministic=True):
    from scann_b200.configs import get_config
    from scann_b200.model import create_model
    cfg = get_config(cfg_name)
    cfg["model"]["n_attention"] = n_attention
    cfg["model"].update(over or {})
    return create_model(cfg, seed=seed, deterministic=deterministic)


def _buffers(b):
    out = {k: getattr(b, k).clone() for k in ("atomic", "atom_mask", "nbr", "nmask", "weight", "dist", "target")}
    if b.ring is not None:
        out["ring"] = b.ring.clone()
    return out


def _same_bits(x, y):
    return x.dtype == y.dtype and np.array_equal(x.view(np.uint8) if x.dtype != bool else x,
                                                 y.view(np.uint8) if y.dtype != bool else y)


@pytest.mark.gpu
def test_gathered_buffers_equal_the_host_route_for_three_shuffled_epochs():
    import torch
    from scann_b200.datagenerator import DataIterator, DeviceDataIterator
    de, dn = ragged_set(300, seed=5, use_ring=True)
    host = DataIterator(de, dn, batch_size=64, shuffle=True, use_ring=True, converter=True, g_update=True)
    dev = DeviceDataIterator.from_data_iterator(host)
    eng = _model(NOUP_RING).engine
    assert len(dev) == 5 and 300 % 64
    for ep in range(3):
        assert np.array_equal(host.indexes, dev.indexes)
        for i in range(len(host)):
            bh = eng.load_batch_csr(*host.csr_item(i), plan=False)
            want = _buffers(bh)
            bd = eng.load_batch_gather(dev, *dev.batch_shape(i), plan=False)
            assert bd is bh and bd.h2d_bytes == 0
            got = _buffers(bd)
            for k in want:
                assert torch.equal(got[k].view(torch.uint8), want[k].view(torch.uint8)), (ep, i, k)
            if ep == 0:
                (ih, th), (id_, td) = host[i], dev[i]
                assert ih.keys() == id_.keys() and _same_bits(th, td)
                for k in ih:
                    assert _same_bits(ih[k], id_[k]), k
                (ch, eh), (cd, ed) = host.csr_item(i), dev.csr_item(i)
                assert ch.keys() == cd.keys() and _same_bits(eh, ed)
                for k in ch:
                    assert (ch[k] == cd[k]) if k in ("M", "N") else _same_bits(np.asarray(ch[k]), np.asarray(cd[k])), k
        np.random.seed(100 + ep)
        host.on_epoch_end()
        np.random.seed(100 + ep)
        dev.on_epoch_end()
    eng.check_status()


def _targets(n, seed=0):
    return np.random.default_rng(seed).standard_normal(n).tolist()


@pytest.mark.gpu
@pytest.mark.parametrize("angle", [True, False])
@pytest.mark.parametrize("d_t,w_t", [(4.0, 0.4), (6.0, 0.2)])
def test_from_structures_equals_the_data_iterator_over_voronoi_lists(monkeypatch, angle, d_t, w_t):
    from scann_b200 import model as Mo
    from scann_b200 import voronoi as V
    from scann_b200.datagenerator import DataIterator, DeviceDataIterator
    structs = [s for _, s in _gpu_cases()] + qm9_like(40, seed=9)
    y = _targets(len(structs))
    monkeypatch.setattr(Mo, "_CHUNK_ATOMS", 400)           # several chunks: their CSR is joined on the device
    assert len(Mo._structure_chunks([len(s.atomic_numbers) for s in structs], 32)) > 1
    dev = DeviceDataIterator.from_structures(structs, y, batch_size=32, g_update=angle, d_t=d_t, w_t=w_t,
                                             converter=True)
    de = np.empty(len(structs), object)
    for k, (s, t) in enumerate(zip(structs, y)):
        de[k] = (list(s.atomic_numbers), t)
    dn = np.empty(len(structs), object)
    for k, lists in enumerate(V.compute_voronoi_neighbors(structs, d_t, w_t)):
        dn[k] = lists
    host = DataIterator(de, dn, batch_size=32, g_update=angle, converter=True)
    assert len(dev) == len(host) and dev.weight_index == host.weight_index
    for i in range(len(host)):
        (ch, eh), (cd, ed) = host.csr_item(i), dev.csr_item(i)
        assert _same_bits(eh, ed) and ch["M"] == cd["M"] and ch["N"] == cd["N"]
        for k in ("struct_atom_off", "atom_nbr_off", "z", "nbr_idx", "nbr_w", "nbr_d"):
            assert _same_bits(np.asarray(ch[k]), np.asarray(cd[k])), (i, k)
    (ih, _), (id_, _) = host[0], dev[0]
    for k in ih:
        assert _same_bits(ih[k], id_[k]), k


def _state_equal(a, b):
    return a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2:] == b[2:]


def _fit(route, de, dn, over, epochs=3, deterministic=True, ring=False):
    from scann_b200.datagenerator import DataIterator, DeviceDataIterator
    g_update = (over or {}).get("g_update", True)
    np.random.seed(21)
    it = DataIterator(de[:192], dn[:192], batch_size=32, shuffle=True, g_update=g_update, use_ring=ring)
    vit = DataIterator(de[192:], dn[192:], batch_size=32, g_update=g_update, use_ring=ring)
    if route == "device":
        it, vit = DeviceDataIterator.from_data_iterator(it), DeviceDataIterator.from_data_iterator(vit)
    m = _model(over, deterministic=deterministic)
    m.compile(optimizer=5e-4)
    hist = m.fit(it, epochs=epochs, validation_data=vit, verbose=0)
    eng = m.engine
    return {"hist": hist.history, "params": eng.params.cpu().numpy(), "m": eng.adam_m.cpu().numpy(),
            "v": eng.adam_v.cpu().numpy(), "rng": np.random.get_state(), "captures": eng.graph_captures,
            "evictions": eng.shape_class_evictions, "dropout": eng.train_dropout}


@pytest.mark.gpu
@pytest.mark.parametrize("over,ring", [(None, False), (NOUP_RING, True)], ids=["qm9", "noupdate_ring"])
def test_fit_gives_the_same_bits_on_both_routes(over, ring):
    de, dn = ragged_set(256, seed=8, use_ring=ring)
    h, d = _fit("host", de, dn, over, ring=ring), _fit("device", de, dn, over, ring=ring)
    assert h["dropout"] and d["dropout"]
    assert h["hist"] == d["hist"] and len(d["hist"]["val_mae"]) == 3
    for k in ("params", "m", "v"):
        assert np.array_equal(h[k].view(np.uint32), d[k].view(np.uint32)), k
    assert _state_equal(h["rng"], d["rng"])
    assert (h["captures"], h["evictions"]) == (d["captures"], d["evictions"])


@pytest.mark.gpu
def test_default_mode_routes_agree_within_the_parity_tolerance():
    de, dn = ragged_set(256, seed=8)
    h = _fit("host", de, dn, None, epochs=1, deterministic=False)
    d = _fit("device", de, dn, None, epochs=1, deterministic=False)
    for k in ("loss", "mae", "val_mae"):
        assert abs(h["hist"][k][0] - d["hist"][k][0]) <= 1e-4 * abs(h["hist"][k][0]), k


@pytest.mark.gpu
def test_prepare_structures_trains_and_evaluates_like_prepare_dataset(tmp_path, monkeypatch):
    from scann_b200 import voronoi as V
    from scann_b200.configs import get_config
    from scann.models import SCANN
    monkeypatch.setenv("TF_DETERMINISTIC_OPS", "1")
    structs = qm9_like(80, seed=12)
    y = _targets(len(structs), seed=3)
    recs = np.empty(len(structs), object)
    for k, (s, t) in enumerate(zip(structs, y)):
        recs[k] = {"Atomic": list(s.atomic_numbers), "Properties": {"homo": t}, "Features": {}}
    nbrs = np.empty(len(structs), object)
    for k, lists in enumerate(V.compute_voronoi_neighbors(structs)):
        nbrs[k] = lists
    np.save(tmp_path / "data.npy", recs, allow_pickle=True)
    np.save(tmp_path / "nbr.npy", nbrs, allow_pickle=True)

    def run(name, prepare):
        cfg = get_config("qm9")
        cfg["model"]["n_attention"] = 2
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
    rep_d, hist_d, sd = run("device", lambda s: s.prepare_structures(structs, y))
    assert sh.config["hyper"]["target_mean"] == sd.config["hyper"]["target_mean"]
    assert sh.config["hyper"]["target_std"] == sd.config["hyper"]["target_std"]
    assert sh.config["hyper"]["data_size"] == sd.config["hyper"]["data_size"] == len(structs)
    assert type(sd.testIter).__name__ == "DeviceDataIterator"
    assert rep_h == rep_d
    assert list(hist_h[0]) == list(hist_d[0]) and list(hist_h[1]) == list(hist_d[1]) and hist_h[2] == hist_d[2]


@pytest.mark.gpu
def test_prepare_structures_refuses_ring_models():
    from scann_b200.configs import get_config
    from scann.models import SCANN
    cfg = get_config("qm9")
    cfg["model"].update(n_attention=2, use_ring=True)
    s = SCANN(cfg, mode="train")
    with pytest.raises(NotImplementedError, match="openbabel"):
        s.prepare_structures(qm9_like(4), [0.0] * 4)
