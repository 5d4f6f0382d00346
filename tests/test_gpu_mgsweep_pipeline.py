"""mgsweep.cuh: the two level sweeps on the shapes where a row pipeline goes wrong.

Each sweep marches a CTA up a band of rows with its loads issued ahead of the arithmetic and its rows kept in
shared-memory rings.  Rows before a band, past its end and off the lattice must read as 0 however short the band or
narrow the strip, and a ring row must not be overwritten while it is still read.  Every case solves with the sweeps and
with the per-kernel path (FEMO_NO_MGSWEEP=1), which must agree bit for bit with equal iteration counts.

FEMO_MGFUSED_MAX_ROWS is lowered so that small lattices put several levels on the sweeps.  Tiles are 128 threads
(122 owned columns + 2 x 3 halo).  Bands are sized to about one wave of resident CTAs and may be one coarse row high;
on a B200 (148 SMs, 8 down-sweep CTAs per SM) a strip gets 1184 / strips bands:
  * 243 x 1201 nodes: two strips, bands of 2 coarse rows and a last band of 1 (601 coarse rows), then 1-row bands;
  * 129 x 401 nodes: two strips, bands of one coarse row on every level;
  * 121 x 201 nodes: one strip whose tile uses all 128 threads;
  * 243 x 201 nodes: two strips of 122 owned columns, the second clipped to 121.
"""
import os

import numpy as np
import pytest

from _cases import Case

pytestmark = pytest.mark.gpu
MAX_ROWS = '500'          # levels above 500 rows take the sweeps (default: 20 000)


def _solve(famid, nx, ny, sweep, graph=False, transpose=False):
    env = {'FEMO_MGFUSED_MAX_ROWS': MAX_ROWS}
    if not sweep:
        env['FEMO_NO_MGSWEEP'] = '1'
    if not graph:
        env['FEMO_NO_GRAPH'] = '1'
    os.environ.update(env)
    try:
        c = Case(famid, nx, ny, seed=7, mg=True, oracle=False)
        if famid == 1:
            _, vals = c.p.assemble_jacobian(plain=False, bc=True)
        else:
            vals, _ = c.p.assemble_jacobian(plain=True, bc=False)
        b = c.p.to_device(np.random.default_rng(13).standard_normal(c.p.N))
        x, info = c.p.linear_solve(vals, b, transpose=transpose, rtol=1e-11, precond=2, cheb_degree=2)
        visits = c.p.vcycle_op_probe(6)[1] if sweep else None     # fine-level down sweeps so far
        return x.cpu().numpy(), info, visits
    finally:
        for k in env:
            os.environ.pop(k, None)


def _check(famid, nx, ny, **kw):
    new = _solve(famid, nx, ny, True, **kw)
    old = _solve(famid, nx, ny, False, **kw)
    assert new[2] >= 2, 'the fine level did not take the sweeps'
    assert new[1]['converged'] and old[1]['converged']
    assert new[1]['iterations'] == old[1]['iterations'], (new[1], old[1])
    assert np.array_equal(new[0], old[0])


@pytest.mark.parametrize('famid', [1, 2])
def test_short_bands(cuda_device, famid):
    """Bands of 2 coarse rows with a last band of 1, and bands of 1: shorter than a band's warm-up.
    Family 1 with Dirichlet masks on both levels of each sweep, family 2 (Nitsche) without."""
    _check(famid, 242, 1200)


@pytest.mark.parametrize('nx', [120, 242])
def test_full_width_tiles(cuda_device, nx):
    """Tiles that use all 128 threads: one strip, and two strips of equal width."""
    _check(2, nx, 200)


@pytest.mark.parametrize('famid', [1, 2])
def test_transposed_solve(cuda_device, famid):
    """Transposed solve: the fine level's planes are converted through t_perm."""
    _check(famid, 128, 400, transpose=True)


def test_graph_replay(cuda_device):
    """The PCG iteration captured into a CUDA graph, with the sweeps recorded in it."""
    _check(2, 242, 200, graph=True)
