"""The dependency-free HDF5 reader/writer (scann_b200/h5lite.py) behind ``load_weights("*.h5")``.

Pin: a file written by libhdf5 itself.  ``tests/golden/testhdf5_7.4_GLNX86.mat`` is a MATLAB v7.3 test file from
SciPy's test data (scipy/io/matlab/tests/data, BSD-3-Clause, see tests/golden/LICENSE.scipy): HDF5 with a 512-byte user block, superblock 0,
symbol-table groups, contiguous float64 dataset, fixed-length string attribute -- the same classic structures h5py
produces for Keras weight files."""
import os

import numpy as np
import pytest

from scann_b200 import h5lite


def _matlab_file():
    return os.path.join(os.path.dirname(__file__), "golden", "testhdf5_7.4_GLNX86.mat")


def test_reads_a_file_written_by_libhdf5():
    f = h5lite.File(_matlab_file())
    assert f.keys() == ["testdouble"]
    d = f["testdouble"]
    assert d.shape == (9, 1) and d.dtype == np.float64
    np.testing.assert_allclose(np.asarray(d).ravel(), np.linspace(0, 2 * np.pi, 9), rtol=1e-15)
    assert d.attrs["MATLAB_class"] == b"double"


def test_keras_layout_round_trip(tmp_path):
    rng = np.random.default_rng(0)
    layers = [("input_1", []),
              ("embed_atom", [("embed_atom/embeddings:0", rng.standard_normal((10, 48)).astype(np.float32))]),
              ("local_attention", [("local_attention/query/kernel:0", rng.standard_normal((128, 128)).astype(np.float32)),
                                   ("local_attention/query/bias:0", rng.standard_normal(128).astype(np.float32))]),
              ("predict_property", [("predict_property/kernel:0", rng.standard_normal((128, 1)).astype(np.float32)),
                                    ("predict_property/bias:0", np.zeros(1, np.float32))])]
    for full in (True, False):
        p = str(tmp_path / f"w{int(full)}.h5")
        h5lite.save_keras_weights(p, layers, full_model=full, model_config='{"class_name": "Functional"}' if full else None)
        back = h5lite.load_keras_weights(p)
        assert [n for n, _ in back] == [n for n, _ in layers]
        for (_, a), (_, b) in zip(layers, back):
            assert [n for n, _ in a] == [n for n, _ in b]
            for (_, x), (_, y) in zip(a, b):
                assert y.dtype == np.float32 and np.array_equal(x, y)
        f = h5lite.File(p)
        assert f.attrs["keras_version"] == b"2.10.0" and f.attrs["backend"] == b"tensorflow"
        if full:
            assert f.attrs["model_config"] == b'{"class_name": "Functional"}'
            assert "model_weights" in f and "embed_atom" in f["model_weights"]


def test_many_links_and_nested_groups(tmp_path):
    w = h5lite.Writer()
    for i in range(100):
        w.dataset(f"/g/sub{i % 7}/d{i}", np.full((3,), i, np.int32))
    w.attr("/g", "names", np.array([b"a", b"bcd", b""]))
    p = str(tmp_path / "n.h5")
    w.save(p)
    f = h5lite.File(p)
    assert sorted(f["g"].keys()) == sorted(f"sub{i}" for i in range(7))
    for i in range(100):
        assert np.array_equal(np.asarray(f[f"g/sub{i % 7}/d{i}"]), np.full((3,), i, np.int32))
    assert list(f["g"].attrs["names"]) == [b"a", b"bcd", b""]


def test_rejects_what_it_does_not_implement(tmp_path):
    p = tmp_path / "x.h5"
    p.write_bytes(b"not hdf5 at all" * 100)
    with pytest.raises(h5lite.H5Error):
        h5lite.File(str(p))
    w = h5lite.Writer()
    w.attr("/", "big", b"x" * 70000)
    with pytest.raises(h5lite.H5Error):
        w.save(str(tmp_path / "y.h5"))
