"""Voronoi neighbour lists (``compute_voronoi_neighbor``, scann/utils/voronoi_neighbor.py:11-61 of the reference).

CPU: the scipy/Qhull oracle (oracle/voronoi_oracle.py) against facts that do not depend on pymatgen -- analytic
lattices, closed cells (solid angles sum to 4 pi, volumes tile the cell, shared facets agree from both sides), the
retry path of a boxed C60, and the hand-over to ``DataIterator`` / ``prepare_input_pmt``.  Where SCANN_REFERENCE_ROOT
names a checkout, the reference's own ``compute_voronoi_neighbor`` runs over a ``VoronoiNN`` stand-in built on the
oracle.  GPU: ``scann_voronoi_neighbors`` (csrc/voronoi.cu) against the oracle."""
import math
import types

import numpy as np
import pytest

from oracle import voronoi_oracle as VO
from tests import ref_stubs

FOUR_PI = 4 * math.pi
PHI = (1 + 5 ** 0.5) / 2


def struct(L, X, Z=None):
    X = np.asarray(X, np.float64)
    return types.SimpleNamespace(lattice=types.SimpleNamespace(matrix=np.asarray(L, np.float64)), cart_coords=X,
                                 atomic_numbers=tuple(Z) if Z is not None else (6,) * len(X))


def fcc(a=4.0):
    return struct(np.eye(3) * a, np.array([[0, 0, 0], [0, .5, .5], [.5, 0, .5], [.5, .5, 0]]) * a)


def analytic():
    a = 3.6
    hcp_L = np.array([[a, 0, 0], [-a / 2, a * 3 ** 0.5 / 2, 0], [0, 0, a * (8 / 3) ** 0.5]])
    hcp = struct(hcp_L, np.array([[1 / 3, 2 / 3, 0.25], [2 / 3, 1 / 3, 0.75]]) @ hcp_L)
    f = np.array([[0, 0, 0], [0, .5, .5], [.5, 0, .5], [.5, .5, 0]])
    rocksalt = struct(np.eye(3) * 5.64, np.concatenate([f, f + 0.5]) * 5.64, [11] * 4 + [17] * 4)
    diamond = struct(np.eye(3) * 3.57, np.concatenate([f, f + 0.25]) * 3.57)
    return {"sc": struct(np.eye(3) * 3.0, [[0, 0, 0]]), "fcc": fcc(),
            "bcc": struct(np.eye(3) * 3.3, np.array([[0, 0, 0], [.5, .5, .5]]) * 3.3),
            "hcp": hcp, "rocksalt": rocksalt, "diamond": diamond}


def c60(box=20.0):
    pts = []
    for base in ((0, 1, 3 * PHI), (1, 2 + PHI, 2 * PHI), (PHI, 2, 2 * PHI + 1)):
        for sx in (1, -1):
            for sy in (1, -1):
                for sz in (1, -1):
                    v = (base[0] * sx, base[1] * sy, base[2] * sz)
                    for r in range(3):
                        pts.append(v[r:] + v[:r])
    X = np.unique(np.round(np.array(pts, np.float64), 12), axis=0) * 0.7 + box / 2     # C-C bond 1.4 Angstrom
    assert len(X) == 60
    return struct(np.eye(3) * box, X)


def random_cell(rng, n, angle=None):
    """Triclinic cell with n sites at least 1 Angstrom apart (periodically)."""
    while True:
        lengths = rng.uniform(3.0, 7.0, 3) * max(1.0, (n / 4) ** (1 / 3))
        al, be, ga = np.radians(rng.uniform(65, 115, 3)) if angle is None else np.radians([90, 90, angle])
        cx = math.cos(be)
        cy = (math.cos(al) - math.cos(be) * math.cos(ga)) / math.sin(ga)
        L = np.array([[lengths[0], 0, 0], [lengths[1] * math.cos(ga), lengths[1] * math.sin(ga), 0],
                      [lengths[2] * cx, lengths[2] * cy, lengths[2] * math.sqrt(max(1 - cx * cx - cy * cy, 1e-3))]])
        F = rng.random((n, 3))
        ok = True
        for i in range(n):
            d = (F - F[i] + 0.5) % 1.0 - 0.5
            r = np.linalg.norm(d @ L, axis=1)
            r[i] = np.inf
            if n > 1 and r.min() < 1.0:
                ok = False
                break
        if ok and np.linalg.norm(L, axis=1).min() >= 1.5:
            return struct(L, F @ L)


def molecule(rng, n, box=20.0):
    """A QM9-sized cluster (atoms at least 1 Angstrom apart in a ~3 Angstrom ball) in a cubic box."""
    X = []
    while len(X) < n:
        p = rng.normal(size=3) * 1.6
        if all(np.linalg.norm(p - q) >= 1.0 for q in X):
            X.append(p)
    return struct(np.eye(3) * box, np.array(X) + box / 2, rng.choice([1, 6, 7, 8, 9], n))


def closed_cells(s):
    L, X = np.asarray(s.lattice.matrix), np.asarray(s.cart_coords)
    return [VO.voronoi_polyhedron(L, X, i) for i in range(len(X))]


# ------------------------------------------------------------------------------------------------ CPU: the oracle
def test_simple_cubic_six_facets_of_two_thirds_pi():
    poly = closed_cells(analytic()["sc"])[0]
    assert len(poly) == 6
    for f in poly:
        assert abs(f["solid_angle"] - 2 * math.pi / 3) < 1e-12 and abs(f["distance"] - 3.0) < 1e-12


def test_fcc_twelve_facets_of_one_third_pi():
    for poly in closed_cells(fcc()):
        big = [f for f in poly if f["normalized"] >= 1e-9]
        assert len(big) == 12
        for f in big:
            assert abs(f["solid_angle"] - math.pi / 3) < 1e-12 and abs(f["distance"] - 4.0 / 2 ** 0.5) < 1e-12


def test_bcc_eight_hexagons_and_six_squares():
    for poly in closed_cells(analytic()["bcc"]):
        assert len(poly) == 14
        d = np.array(sorted(f["distance"] for f in poly))
        assert np.allclose(d[:8], 3.3 * 3 ** 0.5 / 2) and np.allclose(d[8:], 3.3)
        assert sum(f["solid_angle"] for f in poly) == pytest.approx(FOUR_PI, abs=1e-12)


@pytest.mark.parametrize("name", ["hcp", "rocksalt", "diamond"])
def test_closed_cells_cover_the_sphere(name):
    for poly in closed_cells(analytic()[name]):
        assert abs(sum(f["solid_angle"] for f in poly) - FOUR_PI) < 1e-9


def test_random_triclinic_cells_close_and_tile():
    rng = np.random.default_rng(11)
    for t in range(6):
        s = random_cell(rng, int(rng.integers(1, 7)), angle=30.0 if t == 0 else None)
        L = np.asarray(s.lattice.matrix)
        polys = closed_cells(s)
        vol = 0.0
        for i, poly in enumerate(polys):
            assert abs(sum(f["solid_angle"] for f in poly) - FOUR_PI) < 1e-9
            vol += sum(f["volume"] for f in poly)
            for f in poly:                       # the same facet seen from the other side: site i via image -n
                back = [g for g in polys[f["site_index"]] if g["site_index"] == i and g["image"] == tuple(-v for v in f["image"])]
                assert len(back) == 1 and abs(back[0]["area"] - f["area"]) <= 1e-9 * f["area"]
        assert abs(vol - abs(np.linalg.det(L))) < 1e-9 * abs(np.linalg.det(L))


def test_boxed_c60_retries_at_13_angstrom():
    # No image of the molecule in a 20 Angstrom cube closes a cell within 13 Angstrom: every cell is unbounded and
    # pymatgen's loop widens the cutoff to 26 Angstrom.
    s = c60()
    L, X = np.asarray(s.lattice.matrix), np.asarray(s.cart_coords)
    facets, infinite = VO._cell(L, X, 0, 13.0, False)
    assert infinite and facets is None
    poly = VO.voronoi_polyhedron(L, X, 0)
    assert abs(sum(f["solid_angle"] for f in poly) - FOUR_PI) < 1e-9
    with pytest.raises(ValueError, match="no finite Voronoi facet"):   # allowed: every facet infinite, all dropped
        VO.voronoi_polyhedron(L, X, 0, allow_pathological=True)


def test_no_lattice_and_coincident_sites_raise():
    with pytest.raises(ValueError, match="lattice"):
        VO.compute_voronoi_neighbor(types.SimpleNamespace(cart_coords=np.zeros((2, 3)), lattice=None))
    with pytest.raises(ValueError, match="site 0"):
        VO.compute_voronoi_neighbor(struct(np.eye(3) * 4, [[0, 0, 0], [0, 0, 1e-9]]))


def test_oracle_lists_feed_the_data_iterator_and_prepare_input_pmt():
    from scann.utils import DataIterator, prepare_input_pmt
    rng = np.random.default_rng(3)
    structs = [analytic()["rocksalt"], random_cell(rng, 5)]
    nbrs = [VO.compute_voronoi_neighbor(s) for s in structs]
    for s, nb in zip(structs, nbrs):
        inputs = prepare_input_pmt(s, d_t=4.0, w_t=0.4, angle=False, neighbors=nb)
        assert inputs["neighbors"].shape[:2] == (1, len(s.cart_coords))
        assert inputs["neighbor_mask"].sum() == sum(len(a) for a in nb)
        assert (inputs["neighbor_weight"][inputs["neighbor_mask"]] >= 0.4 - 1e-6).all()
    de = np.empty(2, object)
    dn = np.empty(2, object)
    for k, (s, nb) in enumerate(zip(structs, nbrs)):
        de[k], dn[k] = (list(s.atomic_numbers), 0.5 * k), nb
    batch, _ = DataIterator(de, dn, batch_size=2)[0]
    assert batch["neighbors"].shape[0] == 2 and batch["neighbor_mask"].any()


class _Site:
    def __init__(self, coords, index, image):
        self.coords, self.index, self.image = np.asarray(coords), index, image


class _VoronoiNNStandIn:
    """pymatgen ``VoronoiNN`` on the oracle: the calls a caller of ``weight="solid_angle"`` makes."""

    def __init__(self, tol=0, targets=None, cutoff=13.0, allow_pathological=False, weight="solid_angle", **kw):
        assert weight == "solid_angle" and targets is None
        self.tol, self.cutoff, self.allow_pathological, self.weight = tol, cutoff, allow_pathological, weight

    def _poly(self, structure, n):
        L, X = np.asarray(structure.lattice.matrix), np.asarray(structure.cart_coords)
        return L, X, VO.voronoi_polyhedron(L, X, n, self.cutoff, self.allow_pathological)

    def get_voronoi_polyhedra(self, structure, n):
        L, X, poly = self._poly(structure, n)
        return {k: {"site": _Site(X[f["site_index"]] + np.array(f["image"]) @ L, f["site_index"], f["image"]),
                    "solid_angle": f["solid_angle"], "face_dist": f["distance"] / 2, "area": f["area"],
                    "volume": f["volume"]} for k, f in enumerate(poly)}

    def get_nn_info(self, structure, n):
        L, X, poly = self._poly(structure, n)
        return [{"site": _Site(X[f["site_index"]] + np.array(f["image"]) @ L, f["site_index"], f["image"]),
                 "image": f["image"], "weight": f["normalized"], "site_index": f["site_index"],
                 "poly_info": {"solid_angle": f["solid_angle"], "face_dist": f["distance"] / 2}} for f in poly]

    def get_all_nn_info(self, structure):
        return [self.get_nn_info(structure, n) for n in range(len(structure.cart_coords))]


@pytest.mark.skipif(not ref_stubs.reference_available(), reason=ref_stubs.SKIP_REASON)
def test_reference_compute_voronoi_neighbor_over_the_oracle(monkeypatch):
    """The reference's own ``compute_voronoi_neighbor`` (voronoi_neighbor.py:11-61), unmodified, with pymatgen's
    ``VoronoiNN`` replaced by the oracle stand-in: its lists equal the oracle's up to order."""
    import importlib
    import sys
    ref_stubs.load_reference()
    saved = {k: v for k, v in sys.modules.items() if k == "scann" or k.startswith("scann.")}
    for k in saved:
        del sys.modules[k]
    finder = ref_stubs._StubFinder()
    sys.meta_path.insert(0, finder)
    sys.path.insert(0, ref_stubs.REFERENCE_ROOT)
    try:
        vn = importlib.import_module("scann.utils.voronoi_neighbor")
    finally:
        sys.path.remove(ref_stubs.REFERENCE_ROOT)
        sys.meta_path.remove(finder)
        for k in [k for k in sys.modules if k == "scann" or k.startswith("scann.")]:
            del sys.modules[k]
        sys.modules.update(saved)
    monkeypatch.setattr(vn, "VoronoiNN", _VoronoiNNStandIn)
    s = analytic()["rocksalt"]
    s.__len__ = lambda: len(s.cart_coords)
    got = vn.compute_voronoi_neighbor(s, d_thresh=4.0, w_thresh=0.4)
    want = VO.compute_voronoi_neighbor(s, 4.0, 0.4)
    key = lambda t: (round(t[-1], 9), t[1])                          # noqa: E731
    for g, w in zip(got, want):
        assert sorted(((n[1], round(n[2], 9), round(n[-1], 9)) for n in g)) == \
            sorted(((n[1], round(n[2], 9), round(n[-1], 9)) for n in w)), key


# ------------------------------------------------------------------------------------------------ GPU against the oracle
def _gpu_cases():
    rng = np.random.default_rng(2024)
    cases = list(analytic().items())
    cases.append(("triclinic_30deg", random_cell(rng, 3, angle=30.0)))
    for t in range(200):
        n = 1 if t < 20 else int(rng.integers(1, 9))
        cases.append((f"random{t}", random_cell(rng, n)))
    for n in (16, 32, 64):
        cases.append((f"random_n{n}", random_cell(rng, n)))
    cases.append(("c60", c60()))
    for t in range(6):
        cases.append((f"qm9like{t}", molecule(rng, int(rng.integers(9, 30)))))
    return cases


@pytest.fixture(scope="module")
def gpu_vs_oracle():
    from scann_b200 import voronoi as V
    cases = _gpu_cases()
    structs = [s for _, s in cases]
    gpu = V.voronoi_polyhedra(structs)
    orc = [closed_cells(s) for s in structs]
    return cases, gpu, orc


@pytest.mark.gpu
def test_gpu_polyhedra_match_the_oracle(gpu_vs_oracle):
    cases, gpu, orc = gpu_vs_oracle
    assert len(cases) >= 210
    for (name, _), g_s, o_s in zip(cases, gpu, orc):
        for i, (g, o) in enumerate(zip(g_s, o_s)):
            go = {(int(r["site"]), tuple(int(v) for v in r["image"])): r for r in g if r["normalized"] >= 1e-6}
            oo = {(f["site_index"], f["image"]): f for f in o if f["normalized"] >= 1e-6}
            assert set(go) == set(oo), (name, i, sorted(set(go) ^ set(oo)))
            for k, f in oo.items():
                r = go[k]
                assert abs(r["solid_angle"] - f["solid_angle"]) <= 1e-9 * f["solid_angle"], (name, i, k)
                assert abs(r["normalized"] - f["normalized"]) <= 1e-9, (name, i, k)
                assert abs(r["distance"] - f["distance"]) <= 1e-12, (name, i, k)


@pytest.mark.gpu
def test_gpu_thresholded_lists_match_the_oracle(gpu_vs_oracle):
    from scann_b200 import voronoi as V
    cases, _, _ = gpu_vs_oracle
    structs = [s for _, s in cases]
    got = V.compute_voronoi_neighbors(structs)
    for (name, s), g_s in zip(cases, got):
        o_s = VO.compute_voronoi_neighbor(s)
        for i, (g, o) in enumerate(zip(g_s, o_s)):
            near = lambda n: abs(n[-1] - 4.0) <= 1e-9 or abs(n[3] - 0.4) <= 1e-9     # noqa: E731
            # equal distances of symmetric lattices may round apart differently: order ties by site and solid angle
            key = lambda n: (round(n[4], 9), n[1], round(n[2], 6))                     # noqa: E731
            gk, ok = sorted((n for n in g if not near(n)), key=key), sorted((n for n in o if not near(n)), key=key)
            assert [(n[0], n[1]) for n in gk] == [(n[0], n[1]) for n in ok], (name, i)
            for a, b in zip(gk, ok):
                assert abs(a[2] - b[2]) <= 1e-9 * b[2] and abs(a[3] - b[3]) <= 1e-9 and abs(a[4] - b[4]) <= 1e-12


@pytest.mark.gpu
def test_gpu_is_deterministic_and_pathological_mode_drops_infinite_facets():
    from scann_b200 import voronoi as V
    rng = np.random.default_rng(5)
    structs = [random_cell(rng, 7), c60(), molecule(rng, 20)]
    a, b = V.voronoi_polyhedra(structs), V.voronoi_polyhedra(structs)
    for sa, sb in zip(a, b):
        for x, y in zip(sa, sb):
            assert x.tobytes() == y.tobytes()
    with pytest.raises(ValueError, match="structure 0, site 0: its Voronoi cell has no finite facet"):
        V.voronoi_polyhedra([c60()], allow_pathological=True)     # every facet infinite, all dropped


@pytest.mark.gpu
def test_gpu_coincident_sites_raise_naming_structure_and_site():
    from scann_b200 import voronoi as V
    good = analytic()["bcc"]
    bad = struct(np.eye(3) * 4.0, [[0, 0, 0], [1, 1, 1], [1, 1, 1 + 1e-10]])
    with pytest.raises(ValueError, match=r"structure 1, site 1: two points"):
        V.compute_voronoi_neighbors([good, bad])
    with pytest.raises(ValueError, match="lattice"):
        V.compute_voronoi_neighbors([types.SimpleNamespace(cart_coords=np.zeros((2, 3)))])
    assert len(V.compute_voronoi_neighbors([good])[0]) == 2          # the device is still usable


@pytest.mark.gpu
def test_gpu_neighbours_end_to_end_through_prepare_input_pmt_and_predict(tmp_path):
    from scann.models import SCANN
    from scann.utils import compute_voronoi_neighbor, prepare_input_pmt
    from scann_b200.config import model_spec
    from scann_b200.configs import get_config
    from tests.golden.make_golden import oracle_kwargs
    from tests.test_gpu_parity import TOL_OUT, O, rel
    cfg = get_config("qm9")
    cfg["model"]["n_attention"] = 2
    path = str(tmp_path / "w.npz")
    SCANN(cfg, mode="train").model.save_weights(path)
    model = SCANN(cfg, pretrained=path, mode="infer").model
    w = model.engine.get_params()
    from scann_b200.params import ParamLayout
    wd = ParamLayout(model_spec(cfg)).to_dict(w)
    rng = np.random.default_rng(8)
    for s in [molecule(rng, 12), molecule(rng, 21), random_cell(rng, 6)]:
        g_in = prepare_input_pmt(s, d_t=4.0, w_t=0.4, angle=False, neighbors=compute_voronoi_neighbor(s))
        o_in = prepare_input_pmt(s, d_t=4.0, w_t=0.4, angle=False, neighbors=VO.compute_voronoi_neighbor(s))
        for k in o_in:
            assert np.array_equal(g_in[k], o_in[k]) or np.allclose(g_in[k], o_in[k], rtol=1e-6, atol=0), k
        y_g, ga_g = model.predict(g_in)
        y_o, ga_o = model.predict(o_in)
        np.testing.assert_allclose(y_g, y_o, rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(ga_g, ga_o, rtol=1e-6, atol=1e-7)
        y_ref, ga_ref = O.predict(wd, o_in, **oracle_kwargs(model_spec(cfg)))
        assert rel(y_g, y_ref) <= TOL_OUT and rel(ga_g, ga_ref) <= TOL_OUT
