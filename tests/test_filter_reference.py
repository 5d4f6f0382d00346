"""Density filter (SURVEY.md 8f rank 1) held to the reference's own output: tests/golden/filter_reference.npz was produced by
running the reference's examples/beam_topo_opt/pre_processor/general_filter_model.py itself (scripts/make_filter_golden.py).
The oracle's restatement (one KD-tree instead of one per point) must give the same weights and filtered field; the GPU filter
is compared with the oracle's weights in tests/test_gpu_api.py.  No GPU."""
import importlib.util
import os

import numpy as np
import pytest
import scipy.sparse as sp

from oracle.filter import weight_matrix

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, 'golden', 'filter_reference.npz')
CASES = ['lattice2d', 'lattice3d', 'scattered']


def _gen():
    spec = importlib.util.spec_from_file_location('_mk_filter', os.path.join(HERE, '..', 'scripts', 'make_filter_golden.py'))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


@pytest.mark.parametrize('name', CASES)
def test_oracle_filter_equals_the_reference_output(name):
    z = np.load(GOLD)
    coords = z[name + '_coords']
    n = coords.shape[0]
    Wr = sp.csr_matrix((z[name + '_vals'], (z[name + '_rows'], z[name + '_cols'])), shape=(n, n))
    Wo = weight_matrix(coords, float(z[name + '_h_avg']), float(z[name + '_beta']))
    assert (Wr != Wo).nnz == 0 or abs(Wr - Wo).max() <= 1e-15
    assert np.array_equal(Wr.indptr, Wo.indptr) and np.array_equal(Wr.indices, Wo.sorted_indices().indices)
    assert np.abs(Wo @ z[name + '_x'] - z[name + '_y']).max() <= 1e-15
    assert np.abs(np.asarray(Wr.sum(axis=1)).ravel() - 1.0).max() < 1e-14          # rows are partitions of unity


def test_fixture_is_what_the_reference_does_today():
    m = _gen()
    if not m.REF or not os.path.exists(m.REF):
        pytest.skip('no reference checkout')
    live = m.run(m.load_reference_filter())
    z = np.load(GOLD)
    assert sorted(live) == sorted(z.files)
    for k in live:
        assert np.array_equal(np.asarray(live[k]), z[k]), k


@pytest.mark.parametrize('name', ['lattice2d', 'lattice3d'])
def test_mirror_lattice_weights_equal_the_reference_output(name):
    """The product's filter never builds the matrix for its own use: on lattices of cell centres the neighbour offsets and cone
    weights follow from (h, radius) and are applied matrix-free on the device (femo_filter_apply3).  Its HOST-side description
    of the same operator (`weight_triplets`, what real CSDL gets as the constant sparse Jacobian) must be the reference's matrix."""
    from femo_b200.csdl_opt.pre_processor.general_filter_model import GeneralFilterOperation
    z = np.load(GOLD)
    coords = z[name + '_coords']
    n = coords.shape[0]
    op = GeneralFilterOperation(nel=n, beta=float(z[name + '_beta']), coordinates=coords, h_avg=float(z[name + '_h_avg']))
    r, c, v = op.weight_triplets()
    W = sp.csr_matrix((v, (r, c)), shape=(n, n))
    Wr = sp.csr_matrix((z[name + '_vals'], (z[name + '_rows'], z[name + '_cols'])), shape=(n, n))
    assert abs(W - Wr).max() <= 1e-15 and W.nnz == Wr.nnz
    assert np.abs(W @ z[name + '_x'] - z[name + '_y']).max() <= 1e-15
