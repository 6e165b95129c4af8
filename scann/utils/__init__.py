"""``scann.utils`` import path of the reference (scann/utils/__init__.py) on the accelerated package: the data
iterator, the padding helpers, the data-set loaders, and ``compute_voronoi_neighbor`` -- the Voronoi neighbour lists
the model's input is built from, computed on the GPU instead of by pymatgen (``scann_b200/voronoi.py``).  The raw-file
loaders (pymatgen, openbabel) stay outside the package (DESIGN.md section 1)."""
from scann_b200.datagenerator import (DataIterator, load_atomic_features, load_dataset, pad_nested_sequences,  # noqa: F401
                                      pad_sequence, prepare_input_from_neighbors, prepare_input_pmt, set_atomic_features,
                                      split_data)
from scann_b200.voronoi import compute_voronoi_neighbor, compute_voronoi_neighbors  # noqa: F401

__all__ = ["DataIterator", "pad_sequence", "pad_nested_sequences", "split_data", "load_dataset",
           "prepare_input_pmt", "prepare_input_from_neighbors", "set_atomic_features", "load_atomic_features",
           "compute_voronoi_neighbor", "compute_voronoi_neighbors"]
