"""The HDF5 files of --large h5py, checked by an independent byte-level walker of the published
format (tests/hdf5_spec_check.py) that is itself pinned to a file written by the real libhdf5."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import hdf5_spec_check as spec  # noqa: E402

from phyloligo_b200 import io_formats  # noqa: E402


def test_walker_reads_a_file_written_by_libhdf5():
    """MATLAB 7.3 files are HDF5 files behind a 512-byte user block; this one was written by libhdf5 in
    2008 and holds the variable testdouble = 0 : pi/4 : 2 pi.  It is scipy's own test vector for that
    format (scipy/io/matlab/tests/data/testhdf5_7.4_GLNX86.mat, BSD licence), stored unchanged."""
    path = os.path.join(HERE, "golden", "testhdf5_7.4_GLNX86.mat")
    f = spec.H5File(path)
    assert f.base == 512 and f.eof == os.path.getsize(path)
    root = f.root_group()
    assert list(root) == ["testdouble"]
    oh, cache, _ = root["testdouble"]
    got = f.read(oh)
    assert got.dtype == np.float64 and got.shape == (9, 1)
    assert np.array_equal(got[:, 0], np.arange(9) * (np.pi / 4))


@pytest.mark.parametrize("name,shape,dtype", [("distances", (37, 37), np.float32), ("frequencies", (5, 256), np.float32),
                                              ("frequencies", (3, 4096), np.float64), ("distances", (1, 1), np.float32),
                                              ("frequencies", (0, 256), np.float32)])
def test_writer_output_follows_the_specification(tmp_path, name, shape, dtype):
    rng = np.random.default_rng(7)
    arr = rng.random(shape).astype(dtype)
    path = os.path.join(tmp_path, "out.h5")
    io_formats.write_hdf5(path, name, arr)
    f = spec.H5File(path)
    assert f.base == 0 and f.eof == os.path.getsize(path)          # libhdf5: "truncated file" otherwise
    assert (f.leaf_k, f.internal_k) == (4, 16)                      # the library's defaults; node sizes follow from them
    root = f.root_group()
    assert list(root) == [name]
    oh, cache, _ = root[name]
    assert cache == 0
    info = f.dataset(oh)
    assert info["layout"] == "contiguous" and info["layout_version"] == 3 and info["type_version"] == 1
    assert info["shape"] == shape and info["dtype"] == np.dtype(dtype)
    got = f.read(oh)
    assert np.array_equal(got, arr)
    # and the repo's own reader agrees with the walker on where the data is
    shp, dt, addr = io_formats.dataset_location(path, name)
    assert (tuple(shp), np.dtype(dt)) == (shape, np.dtype(dtype))
    if arr.size:
        assert addr == info["address"] and addr % 8 == 0


def test_row_block_writer_and_attach(tmp_path):
    """The file compute_distances_h5py fills: header written first, rows dropped into the data region
    later by other processes -- still a valid file at every step."""
    path = os.path.join(tmp_path, "d.h5")
    w = io_formats.Hdf5DatasetWriter(path, "distances", (50, 50), np.float32)
    w.close()
    f = spec.H5File(path)
    oh = f.root_group()["distances"][0]
    assert not f.read(oh).any()
    a = np.arange(2500, dtype=np.float32).reshape(50, 50)
    with io_formats.Hdf5DatasetWriter.attach(path, "distances") as w2:
        w2.write_rows(10, a[10:30])
    got = spec.H5File(path).read(oh)
    assert np.array_equal(got[10:30], a[10:30]) and not got[:10].any() and not got[30:].any()


def test_walker_rejects_damage(tmp_path):
    path = os.path.join(tmp_path, "x.h5")
    io_formats.write_hdf5(path, "distances", np.ones((4, 4), np.float32))
    good = open(path, "rb").read()
    for pos, why in ((13, "size of offsets"), (40, "end-of-file address"), (140, "root object header")):
        bad = bytearray(good)
        bad[pos] ^= 0xFF
        with pytest.raises((spec.SpecError, ValueError, IndexError, Exception)):
            f = spec.H5File(bytes(bad))
            f.read(f.root_group()["distances"][0])
    with pytest.raises(spec.SpecError):
        spec.H5File(good[:-8])  # truncated: shorter than the end-of-file address
