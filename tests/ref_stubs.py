"""Import the reference's own pure-Python modules (from the checkout of the reference SCANN project that the
environment variable ``SCANN_REFERENCE_ROOT`` names, when it is set) with the third-party packages that are not
installed here replaced by inert stubs.  The reference's source is not part of this repository: without it the tests
that import it skip, while the vectors its graph code produced (``tests/golden/ref_*.npz``) are checked everywhere.

The reference is Python on TensorFlow / Keras / pymatgen / openbabel / ase (SURVEY.md F1, F2); none of them is
installable in this image.  The modules that feed and surround the hot path -- ``scann/utils/datagenerator.py``
(``DataIterator``), ``scann/utils/general.py`` (``pad_sequence``, ``pad_nested_sequences``) and
``scann/layers/custom_layers.py`` (``SGDRC``) -- only need those packages at IMPORT time (base classes, decorators);
their arithmetic is numpy.  A ``sys.meta_path`` finder serves stub modules for the missing roots, the reference tree
is imported under its own top-level name ``scann`` (its modules use absolute ``scann.*`` imports), and this repo's
``scann`` alias package is put back afterwards.  The returned objects are the reference's own functions and
classes, unmodified: a test that compares against them is pinned to reference-run code, not to a restatement.
"""
from __future__ import annotations

import importlib
import importlib.abc
import importlib.machinery
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("SCANN_REFERENCE_ROOT", "")
STUB_ROOTS = ("tensorflow", "keras", "openbabel", "pymatgen", "ase", "tqdm", "h5py", "wget", "requests")
SKIP_REASON = "needs the reference SCANN source: set SCANN_REFERENCE_ROOT to a checkout of it"


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "scann", "utils", "datagenerator.py"))


GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")


def check_stored(name: str, values: dict, rtol: float = 0.0, atol: float = 0.0) -> None:
    """Compares ``values`` (str -> array) with ``tests/golden/reference/<name>.npz``: what a comparison with the
    reference's own code found, so that it keeps being checked where the reference's source is absent.  Where the
    reference is present the calling test also compares the same values with it live, so a stale file cannot pass.
    Exact (dtype and bits) unless a tolerance is given.  ``SCANN_WRITE_REFERENCE_GOLDEN=1`` rewrites the file."""
    import numpy as np
    path = os.path.join(GOLDEN_DIR, name + ".npz")
    values = {k: np.asarray(v) for k, v in values.items()}
    if os.environ.get("SCANN_WRITE_REFERENCE_GOLDEN") == "1":
        os.makedirs(GOLDEN_DIR, exist_ok=True)
        np.savez_compressed(path, **values)
        return
    z = np.load(path)
    assert sorted(z.files) == sorted(values), (name, sorted(set(z.files) ^ set(values)))
    for k, v in values.items():
        assert z[k].dtype == v.dtype and z[k].shape == v.shape, (name, k, z[k].dtype, v.dtype, z[k].shape, v.shape)
        if (rtol or atol) and v.dtype.kind == "f":
            np.testing.assert_allclose(v, z[k], rtol=rtol, atol=atol, err_msg=f"{name}: {k}")
        else:
            assert np.array_equal(v, z[k], equal_nan=v.dtype.kind == "f"), (name, k)


class _StubMeta(type):
    """Module-level constants of stubbed packages (``ase.units.Hartree / eV`` ...) take part in import-time
    arithmetic: every operation on a stub class yields 1.0."""

    def _one(cls, *a):
        return 1.0

    __truediv__ = __rtruediv__ = __mul__ = __rmul__ = __add__ = __radd__ = __sub__ = __rsub__ = __pow__ = _one
    __float__ = _one

    def __getattr__(cls, name):                 # tf.keras.layers.Layer: attribute chains through stub classes
        if name.startswith("__"):
            raise AttributeError(name)
        obj = _StubMeta(name, (_StubBase,), {})
        setattr(cls, name, obj)
        return obj


class _StubBase(metaclass=_StubMeta):
    """Stands in for any class / callable of a stubbed package: subclassable, callable, decorator-friendly."""

    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return self

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _StubBase()


class _StubModule(types.ModuleType):
    __path__: list = []

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        full = self.__name__ + "." + name
        if full in sys.modules:
            return sys.modules[full]
        obj = type(name, (_StubBase,), {"__module__": self.__name__})
        setattr(self, name, obj)
        return obj


class _StubFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def find_spec(self, fullname, path=None, target=None):
        if fullname.split(".")[0] in STUB_ROOTS:
            return importlib.machinery.ModuleSpec(fullname, self, is_package=True)
        return None

    def create_module(self, spec):
        return _StubModule(spec.name)

    def exec_module(self, module):
        pass


_cache = None


def load_reference():
    """-> dict with the reference's own ``DataIterator``, ``pad_sequence``, ``pad_nested_sequences``, ``SGDRC``,
    ``atomic_features`` and the module objects (``datagenerator``, ``general``, ``custom_layers``)."""
    global _cache
    if _cache is not None:
        return _cache
    if not reference_available():
        raise FileNotFoundError(REFERENCE_ROOT)
    saved = {k: v for k, v in sys.modules.items() if k == "scann" or k.startswith("scann.")}
    for k in saved:
        del sys.modules[k]
    finder = _StubFinder()
    really_missing = []
    for root in STUB_ROOTS:
        try:
            importlib.import_module(root)
        except Exception:
            really_missing.append(root)
    sys.meta_path.insert(0, finder)
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        dg = importlib.import_module("scann.utils.datagenerator")
        gen = importlib.import_module("scann.utils.general")
        cl = importlib.import_module("scann.layers.custom_layers")
        ad = importlib.import_module("scann.utils.dataset.atomic_data")
        assert os.path.realpath(dg.__file__).startswith(os.path.realpath(REFERENCE_ROOT))
        _cache = {"DataIterator": dg.DataIterator, "pad_sequence": gen.pad_sequence,
                  "pad_nested_sequences": gen.pad_nested_sequences, "SGDRC": cl.SGDRC,
                  "atomic_features": ad.atomic_features, "datagenerator": dg, "general": gen, "custom_layers": cl,
                  "stubbed": really_missing}
    finally:
        sys.path.remove(REFERENCE_ROOT)
        sys.meta_path.remove(finder)
        for k in [k for k in sys.modules if k == "scann" or k.startswith("scann.") or k.split(".")[0] in really_missing]:
            del sys.modules[k]
        sys.modules.update(saved)
    return _cache


_graph_cache = None


def load_reference_graph():
    """The reference's own GRAPH code on the functional TensorFlow stand-in ``tests/tf_shim.py`` (PyTorch-CPU
    primitives; pymatgen / openbabel / ase ... stay inert stubs).  -> dict with the reference's ``create_model``
    (scann/models/scann_model.py:329-453), ``LocalAttention`` / ``GlobalAttention`` / ``ResidualNorm``
    (scann/layers/attention.py), ``GaussianExpansion`` / ``gather_shape`` / ``mrelu`` (scann/layers/custom_layers.py),
    ``root_mean_squared_error`` (scann/layers/losses.py) and the shim module (``shim.session(...)`` runs them)."""
    global _graph_cache
    if _graph_cache is not None:
        return _graph_cache
    if not reference_available():
        raise FileNotFoundError(REFERENCE_ROOT)
    from tests import tf_shim
    saved = {k: v for k, v in sys.modules.items()
             if k == "scann" or k.startswith("scann.") or k == "tensorflow" or k.startswith("tensorflow.")}
    for k in saved:
        del sys.modules[k]
    finder = _StubFinder()
    really_missing = []
    for root in STUB_ROOTS:
        if root == "tensorflow":
            continue
        try:
            importlib.import_module(root)
        except Exception:
            really_missing.append(root)
    sys.modules.update(tf_shim.build_modules())
    sys.meta_path.insert(0, finder)
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        sm = importlib.import_module("scann.models.scann_model")
        att = importlib.import_module("scann.layers.attention")
        cl = importlib.import_module("scann.layers.custom_layers")
        ls = importlib.import_module("scann.layers.losses")
        for m in (sm, att, cl, ls):
            assert os.path.realpath(m.__file__).startswith(os.path.realpath(REFERENCE_ROOT))
        _graph_cache = {"create_model": sm.create_model, "scann_model": sm, "attention": att, "custom_layers": cl,
                        "LocalAttention": att.LocalAttention, "GlobalAttention": att.GlobalAttention,
                        "ResidualNorm": att.ResidualNorm, "GaussianExpansion": cl.GaussianExpansion,
                        "gather_shape": cl.gather_shape, "mrelu": cl.mrelu,
                        "root_mean_squared_error": ls.root_mean_squared_error, "r2_square": ls.r2_square, "SCANN": sm.SCANN, "SGDRC": cl.SGDRC,
                        "shim": tf_shim}
    finally:
        sys.path.remove(REFERENCE_ROOT)
        sys.meta_path.remove(finder)
        for k in [k for k in sys.modules if k == "scann" or k.startswith("scann.") or k == "tensorflow"
                  or k.startswith("tensorflow.") or k.split(".")[0] in really_missing]:
            del sys.modules[k]
        sys.modules.update(saved)
    return _graph_cache
