"""femo_b200/fea/hdf5_lite.py: the pure-Python HDF5 reader behind XDMF meshes with HDF5 heavy data (no GPU, no h5py).

Pinned by a genuine HDF5 file (tests/golden/testhdf5_7.4_GLNX86.mat, a MATLAB 7.3 file copied from SciPy's test data,
BSD-3-Clause, written by the HDF5 library itself: user block, superblock 0, symbol-table group, version-1 object header,
contiguous float64 data) and by files laid out by tests/_hdf5_writer.py for the structures that file does not contain
(nested groups, chunked storage with a two-level B-tree, edge chunks, shuffle + deflate, integer and big-endian types)."""
import os

import numpy as np
import pytest

from femo_b200.fea import hdf5_lite
from _hdf5_writer import write


def test_file_written_by_the_hdf5_library():
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'testhdf5_7.4_GLNX86.mat')
    f = hdf5_lite.File(path)
    assert f.base == 512 and f.keys() == ['testdouble']
    a = f['testdouble']
    assert a.dtype == np.float64 and a.shape == (9, 1)
    assert np.allclose(a.ravel(), np.arange(9) * np.pi / 4, rtol=0, atol=1e-15)     # scipy's own expected content


@pytest.mark.parametrize('kw', [dict(), dict(chunks=(7, 2)), dict(chunks=(5, 3), gzip=4), dict(chunks=(4, 2), gzip=6, shuffle=True),
                                dict(chunks=(3, 3), gzip=1, shuffle=True, two_level=True)])
def test_layouts_and_filters(tmp_path, kw):
    rng = np.random.default_rng(0)
    tree = {'Mesh': {'mesh': {'geometry': rng.standard_normal((23, 3)), 'topology': rng.integers(0, 23, (40, 3)).astype(np.int64)}},
            'data0': rng.standard_normal((17, 2)).astype('<f4'), 'data1': rng.integers(-5, 5, (31, 4)).astype(np.int32),
            'be': rng.standard_normal((6, 2)).astype('>f8'), 'u1': rng.integers(0, 255, (9, 1)).astype(np.uint8)}
    path = str(tmp_path / 'f.h5')
    write(path, tree, **kw)
    f = hdf5_lite.File(path)
    assert f.keys() == ['Mesh', 'be', 'data0', 'data1', 'u1'] and f.keys('/Mesh/mesh') == ['geometry', 'topology']
    for name, a in (('/Mesh/mesh/geometry', tree['Mesh']['mesh']['geometry']), ('Mesh/mesh/topology', tree['Mesh']['mesh']['topology']),
                    ('data0', tree['data0']), ('/data1', tree['data1']), ('be', tree['be']), ('u1', tree['u1'])):
        b = f[name]
        assert b.shape == a.shape and b.dtype.itemsize == a.dtype.itemsize and b.dtype.kind == a.dtype.kind
        assert np.array_equal(b, a)
    with pytest.raises(KeyError):
        f['/Mesh/nothing']


def test_user_block_and_one_dimensional_data(tmp_path):
    path = str(tmp_path / 'u.h5')
    a = np.arange(1000, dtype=np.int64)
    write(path, {'v': a}, userblock=1024, chunks=lambda x: (128,), gzip=4, shuffle=True)
    f = hdf5_lite.File(path)
    assert f.base == 1024 and np.array_equal(f['v'], a)


def test_not_hdf5(tmp_path):
    p = tmp_path / 'x.h5'
    p.write_bytes(b'version https://git-lfs.github.com/spec/v1\noid sha256:00\nsize 31425\n')       # what the reference checkout holds
    with pytest.raises(ValueError):
        hdf5_lite.File(str(p))


def test_xdmf_with_dolfinx_style_items(tmp_path):
    """dolfinx's XDMFFile writes `Format="h5"` items addressing nested groups (/Mesh/<name>/geometry, /topology) and leaves the
    number type of the geometry item out; read_xdmf resolves both through hdf5_lite."""
    from femo_b200.fea.mesh_io import read_xdmf
    pts = np.array([[0.0, 0.0], [1.0, 0.0], [0.0, 1.0], [1.0, 1.0]])
    conn = np.array([[0, 1, 3], [0, 2, 3]], dtype=np.int64)
    write(str(tmp_path / 'm.h5'), {'Mesh': {'Grid': {'geometry': pts, 'topology': conn}}})
    (tmp_path / 'm.xdmf').write_text(
        '<Xdmf Version="3.0"><Domain><Grid Name="Grid" GridType="Uniform">'
        '<Topology TopologyType="Triangle" NumberOfElements="2" NodesPerElement="3">'
        '<DataItem Dimensions="2 3" NumberType="Int" Format="h5">m.h5:/Mesh/Grid/topology</DataItem></Topology>'
        '<Geometry GeometryType="XY"><DataItem Dimensions="4 2" Format="h5">m.h5:/Mesh/Grid/geometry</DataItem></Geometry>'
        '</Grid></Domain></Xdmf>')
    p, (kind, c), vals = read_xdmf(str(tmp_path / 'm.xdmf'))
    assert kind == 'triangle' and vals is None and np.array_equal(p, pts) and np.array_equal(c, conn)


def test_random_round_trips(tmp_path):
    """Seeded sweep over ranks 1 - 3, dtypes, chunk shapes (smaller than, equal to and larger than the array), filters and
    one- / two-level chunk B-trees."""
    rng = np.random.default_rng(7)
    dtypes = ['<f8', '<f4', '<i8', '<i4', '<u2', '>i4', '>f4', '<i1']
    for case in range(60):
        rank = int(rng.integers(1, 4))
        shape = tuple(int(v) for v in rng.integers(1, 9, rank))
        dt = np.dtype(dtypes[int(rng.integers(len(dtypes)))])
        a = (rng.standard_normal(shape) * 100).astype(dt)
        kw = {}
        if rng.random() < 0.75:
            kw['chunks'] = tuple(int(v) for v in rng.integers(1, 11, rank))
            if rng.random() < 0.6:
                kw['gzip'] = int(rng.integers(1, 10))
            kw['shuffle'] = bool(rng.random() < 0.5)
            kw['two_level'] = bool(rng.random() < 0.5)
        path = str(tmp_path / ('r%d.h5' % case))
        write(path, {'g': {'d': a}, 'top': a[..., :1]}, userblock=int(rng.choice([0, 512, 2048])), **kw)
        f = hdf5_lite.File(path)
        for name, ref in (('/g/d', a), ('top', a[..., :1])):
            b = f[name]
            assert b.shape == ref.shape and b.dtype.kind == ref.dtype.kind and b.dtype.itemsize == ref.dtype.itemsize, (case, kw)
            assert np.array_equal(b, ref), (case, shape, dt, kw)
