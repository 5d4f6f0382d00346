"""Golden vectors of the density filter from the REFERENCE ITSELF: imports
$FEMO_REFERENCE/examples/beam_topo_opt/pre_processor/general_filter_model.py (pure numpy / scipy; csdl replaced by femo_b200's
stand-in base classes) and runs its GeneralFilterOperation on a 2-D lattice of cell centres, a 3-D lattice and a scattered
point set.  Stores the weight matrix (COO triplets in the reference's own order) and the filtered field of a seeded density as
tests/golden/filter_reference.npz; tests/test_filter_reference.py holds oracle/filter.py to it.

    FEMO_REFERENCE=<reference checkout> python scripts/make_filter_golden.py
"""
import importlib.util
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = (os.path.join(os.path.abspath(os.environ['FEMO_REFERENCE']), 'examples/beam_topo_opt/pre_processor/general_filter_model.py')
       if os.environ.get('FEMO_REFERENCE') else '')


def load_reference_filter(path=REF):
    from femo_b200.csdl_opt import _csdl_compat as cc
    stub = types.ModuleType('csdl')
    stub.Model, stub.CustomExplicitOperation, stub.custom = cc.Model, cc.CustomExplicitOperation, cc.csdl.custom
    saved = sys.modules.get('csdl')
    sys.modules['csdl'] = stub
    try:
        spec = importlib.util.spec_from_file_location('_ref_general_filter_model', path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        if saved is None:
            sys.modules.pop('csdl', None)
        else:
            sys.modules['csdl'] = saved
    return mod


def cases():
    """name -> (coordinates, h_avg, beta): the cell centres of the example's mesh family (run_topo_opt_cantilever_beam.py:29-34,
    160 x 80 domain), of a hexahedral box, and scattered points."""
    rng = np.random.default_rng(0)
    nx, ny = 12, 7
    hx, hy = 160.0 / nx, 80.0 / ny
    c2 = np.array([[(i + 0.5) * hx, (j + 0.5) * hy] for j in range(ny) for i in range(nx)])
    n3 = (6, 5, 4)
    h3 = (2.0, 2.0, 2.0)
    c3 = np.array([[(i + 0.5) * h3[0], (j + 0.5) * h3[1], (k + 0.5) * h3[2]] for k in range(n3[2]) for j in range(n3[1]) for i in range(n3[0])])
    sc = rng.random((60, 2)) * [4.0, 2.0]
    return dict(lattice2d=(c2, 0.5 * (hx + hy), 2.0), lattice3d=(c3, 2.0, 2.0), scattered=(sc, 0.4, 1.5))


def run(mod):
    out = {}
    rng = np.random.default_rng(1)
    for name, (coords, h_avg, beta) in cases().items():
        nel = coords.shape[0]
        op = mod.GeneralFilterOperation(nel=nel, beta=beta, coordinates=coords, h_avg=h_avg)
        W = op.weight_mtx.tocoo()
        x = rng.random(nel)
        y = {}
        op.compute({'density_unfiltered': x}, y)
        out.update({name + '_coords': coords, name + '_h_avg': np.float64(h_avg), name + '_beta': np.float64(beta),
                    name + '_rows': W.row.astype(np.int32), name + '_cols': W.col.astype(np.int32), name + '_vals': W.data,
                    name + '_x': x, name + '_y': np.asarray(y['density'])})
    return out


if __name__ == '__main__':
    if not REF:
        sys.exit('set FEMO_REFERENCE to a checkout of the reference femo project')
    path = os.path.join(ROOT, 'tests', 'golden', 'filter_reference.npz')
    np.savez_compressed(path, **run(load_reference_filter()))
    print('->', path)
