"""Set-up and adjoint glue between the Krylov iterations, each against the path it replaced (one switch each):

  * the transposed SpMV, and the fine level's DIA conversion of a transposed multigrid CG solve, read the untransposed
    values through t_perm (FEMO_NO_TRANSPOSE_GATHER=1: permuted copy first);
  * the coarsest-level Gauss-Jordan inverse updates only the rows with a nonzero multiplier (FEMO_NO_BAND_INVERSE=1:
    every row), on the geometric multigrid, the dense preconditioner and the AMG coarse level;
  * the multigrid set-up reads all level bounds in one host read (FEMO_MG_SETUP_SYNC_EACH=1: one read per level).

Each pair computes the same doubles in the same order, so results must agree bit for bit, with the same iteration counts.
Lattices are non-square with widths that are not multiples of 32, and the multigrid hierarchy reaches the cooperative coarse
kernel."""
import contextlib
import os

import numpy as np
import pytest

from _cases import Case, relerr, square_boundary_lists
from femo_b200 import engine as E

pytestmark = pytest.mark.gpu
NX, NY = 600, 424          # 7 levels: 601 x 425 nodes down to 11 x 8


@contextlib.contextmanager
def switch(name):
    if name:
        os.environ[name] = '1'
    try:
        yield
    finally:
        if name:
            os.environ.pop(name, None)


def _jacobian(c, famid):
    if famid == 1:
        return c.p.assemble_jacobian(plain=False, bc=True)[1]
    return c.p.assemble_jacobian(plain=True, bc=False)[0]


def _mg_solve(famid, env, transpose=True, profile=False):
    with switch(env):
        c = Case(famid, NX, NY, seed=5, mg=True, oracle=False)
        vals = _jacobian(c, famid)
        b = c.p.to_device(np.random.default_rng(11).standard_normal(c.p.N))
        x, info = c.p.linear_solve(vals, b, transpose=transpose, rtol=1e-11, precond=2, cheb_degree=2)
        d2h = None
        if profile:            # the same solve again, counting device-to-host copies
            import torch
            from torch.profiler import ProfilerActivity, profile as prof_
            torch.cuda.synchronize()
            with prof_(activities=[ProfilerActivity.CUDA]) as pr:
                x2, info2 = c.p.linear_solve(vals, b, transpose=transpose, rtol=1e-11, precond=2, cheb_degree=2)
                torch.cuda.synchronize()
            assert np.array_equal(x2.cpu().numpy(), x.cpu().numpy()) and info2['iterations'] == info['iterations']
            d2h = sum(1 for e in pr.events() if e.name.startswith('Memcpy') and 'DtoH' in e.name)
        return c, x.cpu().numpy(), info, d2h


def _same(new, old):
    assert new[2]['converged'] and old[2]['converged']
    assert new[2]['iterations'] == old[2]['iterations'], (new[2], old[2])
    assert np.array_equal(new[1], old[1])


@pytest.mark.parametrize('famid', [1, 2])
def test_transposed_solve_gathered_dia_bitwise(cuda_device, famid):
    """Family 1 has Dirichlet rows (symmetric), family 2 a nonsymmetric Jacobian: the gathered conversion must give the
    permuted copy's planes, bounds and hence solution."""
    _same(_mg_solve(famid, None), _mg_solve(famid, 'FEMO_NO_TRANSPOSE_GATHER'))


@pytest.mark.parametrize('famid,transpose', [(1, True), (2, True), (2, False)])
def test_band_inverse_multigrid_bitwise(cuda_device, famid, transpose):
    _same(_mg_solve(famid, None, transpose), _mg_solve(famid, 'FEMO_NO_BAND_INVERSE', transpose))


def test_band_inverse_dense_preconditioner(cuda_device):
    """precond 3 inverts the whole 16 x 13 lattice system (Dirichlet rows included): bitwise against the full sweep, and
    the preconditioned solve against numpy.linalg.inv."""
    res = []
    for env in (None, 'FEMO_NO_BAND_INVERSE'):
        with switch(env):
            c = Case(1, 15, 12, seed=2, oracle=False)
            vals = _jacobian(c, 1)
            bh = np.random.default_rng(3).standard_normal(c.p.N)
            x, info = c.p.linear_solve(vals, c.p.to_device(bh), rtol=1e-14, precond=3)
            res.append((x.cpu().numpy(), info))
    assert np.array_equal(res[0][0], res[1][0]) and res[0][1]['iterations'] == res[1][1]['iterations']
    A = c.csr(0, vals).toarray()
    assert relerr(res[0][0], np.linalg.inv(A) @ bh) < 1e-12


def test_band_inverse_amg_coarse_level(cuda_device):
    res = []
    for env in (None, 'FEMO_NO_BAND_INVERSE'):
        with switch(env):
            c = Case(2, 48, bc=True)
            c.set_state(0.3 * np.sin(3 * c.coords[:, 0]) + 0.1)
            _, vals_bc = c.p.assemble_jacobian(plain=False, bc=True)
            amg = c.p.enable_amg(vals_bc, coarse_size=60).amg
            assert amg['coarsest'] <= 512, amg          # inverted explicitly
            bh = np.random.default_rng(4).standard_normal(c.p.N)
            bh[np.unique(np.concatenate(square_boundary_lists(c.coords)))] = 0.0
            x, info = c.p.linear_solve(vals_bc, c.p.to_device(bh), rtol=1e-10, precond=4, cheb_degree=2)
            assert info['converged'], info
            res.append((x.cpu().numpy(), info))
    assert np.array_equal(res[0][0], res[1][0]) and res[0][1]['iterations'] == res[1][1]['iterations']


@pytest.mark.parametrize('famid', [2, E.FAMILY_NLPOISSON_P2])
def test_transpose_spmv_gather_bitwise(cuda_device, famid):
    """dR/du^T x and dR/dm^T x: the lattice P1 family and the P2 family (no lattice operator)."""
    c = Case(famid, 37, 23, seed=7, oracle=False)
    ops = [(0, c.p.assemble_jacobian(plain=True, bc=False)[0]), (1, c.p.assemble_dRdm(0))]
    rng = np.random.default_rng(8)
    for which, v in ops:
        x = c.p.to_device(rng.standard_normal(c.p.pattern_info(which)['rows']))
        new = c.p.spmv(which, v, x, transpose=True).cpu().numpy()
        with switch('FEMO_NO_TRANSPOSE_GATHER'):
            old = c.p.spmv(which, v, x, transpose=True).cpu().numpy()
        assert np.array_equal(new, old), which
        ref = c.csr(which, v).T @ x.cpu().numpy()
        assert relerr(new, ref) < 1e-13


def test_mg_setup_one_host_read(cuda_device):
    """Same bounds (hence the same bits and iterations) with one device-to-host read per set-up instead of one per level
    below the coarsest: the per-level reads are nlev - 1, the batched one is 1."""
    new = _mg_solve(2, None, profile=True)
    old = _mg_solve(2, 'FEMO_MG_SETUP_SYNC_EACH', profile=True)
    _same(new, old)
    nlev = new[0].p.mg_levels
    assert nlev >= 6
    assert old[3] - new[3] == nlev - 2, (old[3], new[3], nlev)
