"""The wide form of the Voronoi cell search: cells of up to 256 facets (64 vertices per facet) for the sites whose cell
overflows the 64-slot form -- slabs and adsorbates with vacuum, whose surface atoms see the periodic images of the
slab across the vacuum.

A site whose narrow cell search sets only the capacity error runs again, at the same cutoff, in the wide form; every
other site keeps the narrow form's records bit for bit.  The free slot of a cut is the lowest free index in both forms,
so a cell that fits in 64 slots gives the same bits from either form.

Known and not covered here: the slots bound the cell while it is built, not only the final cell.  Points enter in
ascending distance, and until the far side of a vacuum is inserted, every point of the slab below that is inserted
bounds the open cell, so a lone adatom under a wide vacuum can overflow 256 slots although its final cell has fewer
facets (DESIGN.md section 4.6)."""
import numpy as np
import pytest

from oracle import voronoi_oracle as VO
from tests.test_predict_structures import qm9_like
from tests.test_ring_routes import CC, PTGP, SHEETS, _pt_sites, _ring_model, _bits, host_batches, ring_rows
from tests.test_voronoi import _gpu_cases, closed_cells, random_cell, struct


def slab(rng, c, m, sheet=None):
    """A graphene sheet (C-C 1.42 Angstrom, jittered by 0.02 Angstrom) with a Pt cluster of m atoms 2.3 Angstrom above
    it, in a cell of height c: a vacuum of about c - 5 Angstrom between the cluster and the next sheet."""
    a, b = np.sqrt(3) * CC, 3 * CC
    cell = np.array([[0, 0], [a / 2, CC / 2], [a / 2, 1.5 * CC], [0, 2 * CC]])
    nx, ny = sheet or SHEETS[int(rng.integers(len(SHEETS)))]
    L = np.diag([nx * a, ny * b, c])
    xy = (cell[None, None] + np.stack(np.meshgrid(np.arange(nx) * a, np.arange(ny) * b, indexing="ij"),
                                      -1)[:, :, None]).reshape(-1, 2)
    C = np.concatenate([xy, np.full((len(xy), 1), 3.0)], 1) + rng.normal(0, 0.02, (len(xy), 3))
    th = rng.uniform(0, 2 * np.pi)
    rot = np.array([[np.cos(th), -np.sin(th), 0], [np.sin(th), np.cos(th), 0], [0, 0, 1]])
    P = _pt_sites()[:m] @ rot.T + [rng.uniform(0, L[0, 0]), rng.uniform(0, L[1, 1]), 3.0 + 2.3]
    return struct(L, np.concatenate([C, P]) % np.diag(L), [6] * len(C) + [78] * m)


def slabs(seed=0):
    """Clusters of 4 and 7 atoms at c = 15, 20 and 25 Angstrom, and a lone adatom at 15."""
    rng = np.random.default_rng(seed)
    return [slab(rng, c, m) for c in (15.0, 20.0, 25.0) for m in (4, 7)] + [slab(rng, 15.0, 1)]


def flags_of(structs):
    return [np.array([[1, 1] if z == 6 else [0, 0] for z in s.atomic_numbers], np.int64) for s in structs]


def pt_facets(s):
    L, X = np.asarray(s.lattice.matrix), np.asarray(s.cart_coords)
    return [len(VO.voronoi_polyhedron(L, X, i)) for i in range(len(X)) if s.atomic_numbers[i] == 78]


def too_wide():
    """A lone adatom under 55 Angstrom of vacuum: a cell of more than 256 facets."""
    return slab(np.random.default_rng(7), 60.0, 1, (7, 6))


# ------------------------------------------------------------------------------------------------ CPU
def test_the_generator_makes_cells_beyond_64_and_128_facets():
    counts = [pt_facets(s) for s in slabs()]
    every = sum(counts, [])
    assert sum(n > 64 for n in every) >= 5 and max(every) > 100, counts
    rng = np.random.default_rng(1)
    assert min(pt_facets(slab(rng, c, 1))[0] for c in (20.0, 25.0)) > 128      # lone adatoms under more vacuum
    assert pt_facets(too_wide())[0] > 256


def test_each_centre_runs_once_per_round_with_pymatgens_cutoffs(monkeypatch):
    """The retry loop with a stand-in for the launch: centres 3 and 7 overflow the narrow form, and centre 7's cell
    stays unbounded below 30 Angstrom.  Every centre runs once per round; 3 and 7 run wide from the round after their
    overflow, at the same cutoff; 7 then widens 13 -> 26 -> 52 as pymatgen does (the cap is 69.29)."""
    from scann_b200 import voronoi as V
    launches = []

    def fake_run(lat, X, sa_off, atoms, cut, allow_pathological, cap=V._CAP):
        launches.append((cap > V._CAP, [int(a) for a in atoms], [float(c) for c in cut]))
        flags = np.zeros(len(atoms), np.int32)
        for k, (a, c) in enumerate(zip(atoms, cut)):
            if a in (3, 7) and cap == V._CAP:
                flags[k] = V.ERR_CAPACITY
            elif a == 7 and c < 30.0:
                flags[k] = V._INFINITE
        n = (flags == 0).astype(np.int32)
        rec = np.zeros(int(n.sum()), V.FACET)
        rec["solid_angle"], rec["normalized"], rec["distance"], rec["image"] = 1.0, 1.0, 2.0, 512 | 512 << 10 | 512 << 20
        rec["site"] = [int(a) for a, f in zip(atoms, flags) if f == 0]
        return np.concatenate([[0], np.cumsum(n)]).astype(np.int32), flags, rec

    monkeypatch.setattr(V, "_run", fake_run)
    X = np.random.default_rng(0).uniform(0, 40, (10, 3))
    out = V.voronoi_polyhedra([struct(np.eye(3) * 40.0, X, [6] * 10)])
    assert launches == [(False, list(range(10)), [13.0] * 10), (True, [3, 7], [13.0, 13.0]), (True, [7], [26.0]),
                        (True, [7], [52.0])], launches
    assert [int(f["site"][0]) for f in out[0]] == list(range(10))
    monkeypatch.setattr(V, "_CHUNK", 4)
    monkeypatch.setattr(V, "_CHUNK_WIDE", 1)
    parts = V._passes(np.arange(10), np.isin(np.arange(10), [2, 5]))
    assert [(list(p), cap, w) for p, cap, w in parts] == [([0, 1, 3, 4], 64, False), ([6, 7, 8, 9], 64, False),
                                                           ([2], 256, True), ([5], 256, True)]


# ------------------------------------------------------------------------------------------------ GPU
def _all_records(structs, cap):
    """One launch of every site of ``structs`` at cutoff 13 with ``cap`` facet slots -> (off, flags, records)."""
    from scann_b200 import voronoi as V
    lats, xs = V._arrays(structs)
    sa = np.zeros(len(xs) + 1, np.int64)
    np.cumsum([len(x) for x in xs], out=sa[1:])
    lat = np.ascontiguousarray(np.stack(lats).reshape(-1, 9))
    X = np.ascontiguousarray(np.concatenate(xs))
    return V._run(lat, X, sa, np.arange(sa[-1]), np.full(sa[-1], 13.0), False, cap)


@pytest.mark.gpu
def test_narrow_and_wide_forms_give_the_same_bits():
    """Every structure of the existing Voronoi tests, plus MP2018-like crystals: the same records, in the same order,
    from 64 and from 256 slots."""
    rng = np.random.default_rng(11)
    structs = [s for _, s in _gpu_cases()] + [random_cell(rng, int(rng.integers(2, 65))) for _ in range(40)]
    off_n, fl_n, rec_n = _all_records(structs, 64)
    off_w, fl_w, rec_w = _all_records(structs, 256)
    assert not (fl_n & ~1).any()                                 # all fit in the narrow form
    assert np.array_equal(fl_n, fl_w) and np.array_equal(off_n, off_w)
    assert rec_n.tobytes() == rec_w.tobytes()
    assert len(rec_n) > 5000 and (fl_n & 1).any()               # infinite cells (the boxed C60) alike


def _sorted(rec):
    img = np.stack([(rec["image"] >> (10 * k)) & 1023 for k in range(3)], -1)
    return rec[np.lexsort((img[:, 2], img[:, 1], img[:, 0], rec["site"], rec["distance"]))]


@pytest.mark.gpu
def test_sites_that_fit_keep_the_narrow_records():
    from scann_b200 import voronoi as V
    structs = slabs()
    off, fl, rec = _all_records(structs, 64)
    cap = (fl & ~1) == V.ERR_CAPACITY
    assert cap.any() and not (fl & ~1 & ~V.ERR_CAPACITY).any()
    got = [r for per in V.voronoi_polyhedra(structs) for r in per]
    for a in np.flatnonzero(fl == 0):
        g, n = got[a], _sorted(rec[off[a]:off[a + 1]])
        assert len(g) == len(n), a
        for name in ("solid_angle", "normalized", "distance", "site"):
            assert g[name].tobytes() == n[name].tobytes(), (a, name)
    assert max(len(g) for g in got) > 100


@pytest.mark.gpu
def test_slab_cells_match_the_oracle():
    from scann_b200 import voronoi as V
    structs = slabs()
    gpu = V.voronoi_polyhedra(structs)
    for k, s in enumerate(structs):
        for i, (g, o) in enumerate(zip(gpu[k], closed_cells(s))):
            go = {(int(r["site"]), tuple(int(v) for v in r["image"])): r for r in g if r["normalized"] >= 1e-6}
            oo = {(f["site_index"], f["image"]): f for f in o if f["normalized"] >= 1e-6}
            assert set(go) == set(oo), (k, i, sorted(set(go) ^ set(oo)))
            for key, f in oo.items():
                r = go[key]
                assert abs(r["solid_angle"] - f["solid_angle"]) <= 1e-9 * f["solid_angle"], (k, i, key)
                assert abs(r["normalized"] - f["normalized"]) <= 1e-9, (k, i, key)
                assert abs(r["distance"] - f["distance"]) <= 1e-12, (k, i, key)
    got = V.compute_voronoi_neighbors(structs)
    near = lambda n: abs(n[-1] - 4.0) <= 1e-9 or abs(n[3] - 0.4) <= 1e-9        # noqa: E731
    key = lambda n: (round(n[4], 9), n[1], round(n[2], 6))                         # noqa: E731
    for s, g_s in zip(structs, got):
        for i, (g, o) in enumerate(zip(g_s, VO.compute_voronoi_neighbor(s))):
            gk, ok = sorted((n for n in g if not near(n)), key=key), sorted((n for n in o if not near(n)), key=key)
            assert [(n[0], n[1]) for n in gk] == [(n[0], n[1]) for n in ok], i
            for a, b in zip(gk, ok):
                assert abs(a[2] - b[2]) <= 1e-9 * b[2] and abs(a[3] - b[3]) <= 1e-9 and abs(a[4] - b[4]) <= 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("angle", [True, False])
def test_device_csr_equals_the_data_iterator(angle):
    from scann_b200 import voronoi as V
    from tests.test_predict_structures import host_iterator
    structs = slabs() + qm9_like(6, seed=5)
    got = V.select_neighbors(structs, angle=angle).csr()
    want, _ = host_iterator(structs, 4.0, 0.4, angle, len(structs)).csr_item(0)
    assert got["M"] == want["M"] and got["N"] == want["N"] and got["P"] == len(want["nbr_idx"])
    for k in ("struct_atom_off", "atom_nbr_off", "z", "nbr_idx"):
        assert np.array_equal(got[k].cpu().numpy(), np.asarray(want[k], np.int32)), k
    for k in ("nbr_w", "nbr_d"):
        assert np.array_equal(got[k].cpu().numpy().view(np.uint32), want[k].view(np.uint32)), k


@pytest.mark.gpu
def test_predict_structures_on_slabs_equals_the_padded_ring_batches():
    model, _ = _ring_model("ptgp", **PTGP)
    structs = slabs(seed=3)
    flags = flags_of(structs)
    y, ga, la = model.predict_structures(structs, batch_size=4, local_attention=True, ring_aromatic=flags)
    want = host_batches(model, structs, flags, 4)
    assert len(want) == len(structs)
    for k, (y_h, ga_h, la_h) in enumerate(want):
        assert _bits(y[k, 0]) == _bits(y_h), k
        assert np.array_equal(_bits(ga[k]), _bits(ga_h)), k
        assert np.array_equal(_bits(la[k].scores), _bits(la_h)), k
    model.engine.check_status()


@pytest.mark.gpu
def test_from_structures_on_slabs_equals_the_host_route():
    import torch
    from scann_b200 import voronoi as V
    from scann_b200.datagenerator import DataIterator, DeviceDataIterator
    from tests.test_ring_routes import _buffers
    structs = slabs(seed=4)
    flags = flags_of(structs)
    y = np.random.default_rng(0).standard_normal(len(structs)).tolist()
    de, dn = ring_rows(structs, V.compute_voronoi_neighbors(structs), flags, y)
    host = DataIterator(de, dn, batch_size=3, shuffle=False, use_ring=True, converter=True, g_update=False)
    dev = DeviceDataIterator.from_structures(structs, y, batch_size=3, shuffle=False, g_update=False, use_ring=True,
                                             ring_aromatic=flags, converter=True)
    eng = _ring_model("ptgp", n_attention=1, infer=False, **PTGP)[0].engine
    for i in range(len(host)):
        want = _buffers(eng.load_batch_csr(*host.csr_item(i), plan=False))
        got = _buffers(eng.load_batch_gather(dev, *dev.batch_shape(i), plan=False))
        for k in want:
            assert torch.equal(got[k].view(torch.uint8), want[k].view(torch.uint8)), (i, k)
    eng.check_status()


@pytest.mark.gpu
def test_more_than_64_kept_neighbours_and_the_wide_limit_raise():
    from scann_b200 import voronoi as V
    structs = [qm9_like(1, seed=1)[0], slabs()[3]]                # c = 20, a cluster of 7: Pt cells of ~100 facets
    with pytest.raises(ValueError, match=r"structure 6, site \d+: \d+ neighbours kept .*more than the 64") as e:
        V.select_neighbors(structs, d_thresh=100.0, w_thresh=0.0, first_index=5)
    site = int(str(e.value).split("site ")[1].split(":")[0])
    assert structs[1].atomic_numbers[site] == 78
    assert len(V.compute_voronoi_neighbors(structs, 100.0, 0.0)[1][site]) > 64      # the host lists have no limit
    s = too_wide()                                               # a final cell of more than 256 facets
    site = len(s.atomic_numbers) - 1
    with pytest.raises(ValueError, match=rf"structure 0, site {site}: .*256 facets, 64 vertices"):
        V.voronoi_polyhedra([s])
    with pytest.raises(ValueError, match=rf"structure 0, site {site}: .*256 facets, 64 vertices"):
        V.select_neighbors([s])
