"""``scann.utils.voronoi_neighbor`` (reference: scann/utils/voronoi_neighbor.py) -- the neighbour search on the GPU."""
from scann_b200.voronoi import compute_voronoi_neighbor, compute_voronoi_neighbors  # noqa: F401
