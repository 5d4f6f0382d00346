"""mgsweep.cuh: the two fused level sweeps of the V-cycle against the per-kernel path (FEMO_NO_MGSWEEP=1).

The sweeps evaluate the same row expressions as k_dia_apply and the nested transfers, so solutions must agree bit for
bit, with the same iteration counts.  Lattices are non-square, their widths are not multiples of the sweep's strip
width, and two levels sit above the cooperative coarse kernel's range (600 x 424: 255 k and 64 k rows)."""
import os

import numpy as np
import pytest

from _cases import Case
from femo_b200 import engine as E

pytestmark = pytest.mark.gpu
NX, NY = 600, 424
ELIGIBLE = 2              # levels above the cooperative kernel's 20 000 rows: 601 x 425 and 301 x 213 nodes


def _solve(famid, nx, ny, sweep, graph, transpose=False):
    if not sweep:
        os.environ['FEMO_NO_MGSWEEP'] = '1'
    if not graph:
        os.environ['FEMO_NO_GRAPH'] = '1'
    try:
        c = Case(famid, nx, ny, seed=5, mg=True, oracle=False)
        if famid == 1:
            _, vals = c.p.assemble_jacobian(plain=False, bc=True)
        else:
            vals, _ = c.p.assemble_jacobian(plain=True, bc=False)
        b = c.p.to_device(np.random.default_rng(11).standard_normal(c.p.N))
        l0 = c.p.launch_count()
        x, info = c.p.linear_solve(vals, b, transpose=transpose, rtol=1e-11, precond=2, cheb_degree=2)
        launches = c.p.launch_count() - l0
        visits = c.p.vcycle_op_probe(6)[1] if sweep and famid != E.FAMILY_NLPOISSON_P2 else None
        return c, x.cpu().numpy(), info, launches, visits
    finally:
        os.environ.pop('FEMO_NO_MGSWEEP', None)
        os.environ.pop('FEMO_NO_GRAPH', None)


def _same(new, old):
    assert new[2]['converged'] and old[2]['converged']
    assert new[2]['iterations'] == old[2]['iterations'], (new[2], old[2])
    assert np.array_equal(new[1], old[1])


@pytest.mark.parametrize('famid,transpose', [(2, False), (2, True), (1, False)])
def test_sweeps_bitwise_and_launches(cuda_device, famid, transpose):
    """Plain launches (no graph): equal bits and iterations, and 4 launches fewer per eligible level visit (six
    per-level kernels become two sweeps).  Fine-level visits = the full-multigrid start + one per preconditioner
    application; the start visits the E eligible levels E(E+1)/2 times, every application E times."""
    new = _solve(famid, NX, NY, True, False, transpose)
    old = _solve(famid, NX, NY, False, False, transpose)
    _same(new, old)
    fine = new[4]
    assert fine >= 2
    visits = ELIGIBLE * (fine - 1) + ELIGIBLE * (ELIGIBLE + 1) // 2
    assert old[3] - new[3] == 4 * visits, (old[3], new[3], fine)


def test_sweeps_bitwise_under_graph_replay(cuda_device):
    """Default settings: the PCG iteration of this size is captured into a CUDA graph; the sweeps are recorded in it."""
    _same(_solve(2, NX, NY, True, True), _solve(2, NX, NY, False, True))


def test_sweeps_bitwise_p2_pmultigrid(cuda_device):
    """P2 -> P1 p-multigrid: the P1 level 1 (301 x 213 nodes) takes the sweeps."""
    _same(_solve(E.FAMILY_NLPOISSON_P2, 300, 212, True, False), _solve(E.FAMILY_NLPOISSON_P2, 300, 212, False, False))


def test_probe_modes_6_7(cuda_device):
    c = _solve(2, NX, NY, True, False)[0]
    N = c.p.N
    for mode in (6, 7):
        b0, n0 = c.p.vcycle_op_probe(mode)
        b1, n1 = c.p.vcycle_op_probe(mode)
        assert b0 == b1 and b0 > 48 * N and n1 == n0 + 1
