"""CPU ORACLE -- TEST INFRASTRUCTURE ONLY.  Not part of the product path: nothing under ``scann_b200/`` or ``scann/``
imports this module.

Restatement, on ``scipy.spatial.Voronoi`` (Qhull, the library pymatgen calls), of the neighbour lists the reference's
``compute_voronoi_neighbor`` (scann/utils/voronoi_neighbor.py:11-61) builds with pymatgen's
``VoronoiNN(weight="solid_angle", tol=0)``: ``get_voronoi_polyhedra`` (point set within ``cutoff`` of the centre,
one Qhull tessellation per site, the retry loop that widens ``cutoff`` while the cell has an infinite facet) +
``_extract_cell_info`` (solid angle of each facet by pymatgen's fan formula) + ``_extract_nn_info`` (weights
normalised by the largest solid angle, facets with weight 0 dropped), followed by the wrapper's distance / weight
thresholds.  The ``sm_100a`` path is ``scann_b200/voronoi.py`` + ``scann_b200/csrc/voronoi.cu``; tests compare the two.
"""
from __future__ import annotations

import math
from typing import Dict, List

import numpy as np
from scipy.spatial import ConvexHull, Voronoi

COINCIDENT = 1e-8      # two points of the set closer than this (Angstrom): Qhull fails, so does the GPU path


def max_cutoff(L) -> float:
    """pymatgen's cap of the retry loop: the longest of the four cell diagonals, plus 0.01."""
    L = np.asarray(L, np.float64)
    corners = np.array([[1, 1, 1], [-1, 1, 1], [1, -1, 1], [1, 1, -1]], np.float64)
    return float(np.linalg.norm(corners @ L, axis=1).max()) + 0.01


def points_in_sphere(L, X, i: int, cutoff: float):
    """Every periodic image ``x_j + n L`` with ``|x_j + n L - x_i| <= cutoff`` (the centre itself included), sorted by
    distance, then site index, then image.  -> (site [K], image [K,3], displacement from x_i [K,3], distance [K])."""
    L, X = np.asarray(L, np.float64), np.asarray(X, np.float64)
    B = np.linalg.inv(L)
    reach = cutoff * np.linalg.norm(B, axis=0)                 # |fractional coordinate k| <= cutoff * |B[:, k]|
    dfrac = (X - X[i]) @ B
    lo = np.floor((-reach - dfrac).min(0)).astype(int)
    hi = np.ceil((reach - dfrac).max(0)).astype(int)
    grid = np.stack(np.meshgrid(*[np.arange(a, b + 1) for a, b in zip(lo, hi)], indexing="ij"), -1).reshape(-1, 3)
    disp = (X - X[i])[:, None, :] + (grid @ L)[None, :, :]
    dist = np.sqrt((disp * disp).sum(-1))
    j, g = np.nonzero(dist <= cutoff)
    site, image, disp, dist = j, grid[g], disp[j, g], dist[j, g]
    order = np.lexsort((image[:, 2], image[:, 1], image[:, 0], site, dist))
    return site[order], image[order], disp[order], dist[order]


def solid_angle(center, coords) -> float:
    """pymatgen.analysis.local_env.solid_angle: fan of tetrahedra from the first vertex (Van Oosterom-Strackee)."""
    r = [np.subtract(c, center) for c in coords]
    rn = [np.linalg.norm(v) for v in r]
    angle = 0.0
    for k in range(1, len(r) - 1):
        tp = abs(np.dot(r[0], np.cross(r[k], r[k + 1])))
        de = rn[0] * rn[k] * rn[k + 1] + rn[k + 1] * np.dot(r[0], r[k]) + rn[k] * np.dot(r[0], r[k + 1]) \
            + rn[0] * np.dot(r[k], r[k + 1])
        a = (0.5 * math.pi if tp > 0 else -0.5 * math.pi) if de == 0 else math.atan(tp / de)
        angle += (a if a > 0 else a + math.pi) * 2
    return angle


def _cell(L, X, i: int, cutoff: float, allow_pathological: bool):
    """One Qhull tessellation of the points within ``cutoff`` of site i.  -> (facets, has_infinite)."""
    site, image, disp, dist = points_in_sphere(L, X, i, cutoff)
    if len(dist) > 1 and dist[1] < COINCIDENT:
        raise ValueError(f"site {i}: coincident with site {int(site[1])} image {tuple(int(v) for v in image[1])}")
    vor = Voronoi(disp)                                        # the centre is point 0 (distance 0, sorted first)
    # the cell is unbounded exactly when the centre is a vertex of the hull of S; asked directly because Qhull drops
    # the ridges of cospherical point sets (a lone fullerene) instead of marking them with -1
    infinite = bool(len(disp) < 5 or 0 in ConvexHull(disp).vertices)
    if infinite and not allow_pathological:
        return None, True
    facets = []
    for (a, b), vind in vor.ridge_dict.items():
        if 0 not in (a, b):
            continue
        k = b if a == 0 else a
        if -1 in vind:
            infinite = True
            if allow_pathological:
                continue
            return None, True
        verts = vor.vertices[vind]
        vol = sum(abs(np.dot(verts[0], np.cross(verts[m], verts[m + 1]))) / 6.0 for m in range(1, len(verts) - 1))
        d = float(dist[k])
        facets.append({"site_index": int(site[k]), "image": tuple(int(v) for v in image[k]), "distance": d,
                       "solid_angle": solid_angle(np.zeros(3), verts), "volume": vol, "area": 3.0 * vol / (d / 2)})
    return facets, infinite


def voronoi_polyhedron(L, X, i: int, cutoff: float = 13.0, allow_pathological: bool = False) -> List[Dict]:
    """pymatgen ``VoronoiNN.get_voronoi_polyhedra`` + ``_extract_nn_info`` (weight="solid_angle", tol=0) for site i:
    the finite facets with solid angle > 0, each with ``normalized`` = solid angle / the site's largest."""
    top = max_cutoff(L)
    while True:
        facets, infinite = _cell(L, X, i, cutoff, allow_pathological)
        if not infinite or allow_pathological:
            break
        if cutoff >= top:
            raise ValueError(f"site {i}: infinite Voronoi facet at the largest cutoff {cutoff:.3f}")
        cutoff = min(2 * cutoff, top + 0.001)
    if not facets:
        raise ValueError(f"site {i}: no finite Voronoi facet")
    wmax = max(f["solid_angle"] for f in facets)
    kept = [dict(f, normalized=f["solid_angle"] / wmax) for f in facets if f["solid_angle"] > 0]
    kept.sort(key=lambda f: (f["distance"], f["site_index"], f["image"]))
    return kept


def _as_arrays(struct):
    lat = getattr(struct, "lattice", None)
    if lat is None:
        raise ValueError("the structure has no lattice: box a molecule first")
    return np.asarray(lat.matrix, np.float64), np.asarray(struct.cart_coords, np.float64)


def compute_voronoi_neighbor(struct, d_thresh: float = 4.0, w_thresh: float = 0.4, cutoff: float = 13.0,
                             allow_pathological: bool = False):
    """Per atom i, the tuples ``(i, site_index, solid_angle, normalized, distance)`` of the facets with
    ``distance <= d_thresh`` and ``normalized >= w_thresh``, sorted by distance, site index, image."""
    L, X = _as_arrays(struct)
    out = []
    for i in range(len(X)):
        poly = voronoi_polyhedron(L, X, i, cutoff, allow_pathological)
        out.append([(i, f["site_index"], f["solid_angle"], f["normalized"], f["distance"]) for f in poly
                    if f["distance"] <= d_thresh and f["normalized"] >= w_thresh])
    return out
