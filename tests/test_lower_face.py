"""The constants and conventions of the hot path, taken from the REFERENCE'S OWN CODE instead of from memory:
tests/golden/lower_face_calls.json records what femo/fea/utils_dolfinx.py (run unmodified over a recording stand-in for
dolfinx / PETSc, tests/_lower_face.py, scripts/make_lower_face_calls.py) asks the libraries to do.  The oracle
(oracle/solvers.py, oracle/assembly.py) and the product's defaults (femo_b200/engine.py, femo_b200/fea/utils_b200.py) are
compared with that recording.  No GPU."""
import ctypes as C
import inspect
import json
import os

import numpy as np
import pytest

import _lower_face as L

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'lower_face_calls.json')


@pytest.fixture(scope='module')
def ref():
    with open(GOLD) as f:
        return json.load(f)


def _sets(events, suffix):
    return {e[1].rsplit('.', 1)[1]: e[2] for e in events if e[0] == 'set' and suffix in e[1]}


def _calls(events, name):
    return [e for e in events if e[0] == 'call' and e[1].endswith(name)]


def test_fixture_is_what_the_reference_does_today(ref):
    if not L.REFERENCE or not os.path.isdir(os.path.join(L.REFERENCE, 'femo')):
        pytest.skip('no reference checkout')
    assert json.loads(json.dumps(L.record())) == ref


def _engine_newton_opts(kind):
    """The femo_newton_opts struct EngineProblem.newton_solve hands to the C ABI with its defaults."""
    from femo_b200 import engine as E
    seen = {}

    class Spy:
        def __getattr__(self, k):
            def f(h, opts, info):
                o = opts._obj
                seen.update(kind=o.kind, atol=o.atol, rtol=o.rtol, stol=o.stol, max_it=o.max_it)
                return 0
            return f
    p = object.__new__(E.EngineProblem)
    p._h = None
    lib, E.lib = E.lib, Spy()
    try:
        p.newton_solve(kind=kind)
    finally:
        E.lib = lib
    return seen


def test_newton_solver_constants(ref):
    """utils_dolfinx.py:419-449 as executed: atol 1e-50, rtol 1e-30, max_it 3, error_on_nonconvergence False -> three Newton steps,
    never an error (quirk B1); `initialize` presets the state to 0.1."""
    s = _sets(ref['NewtonSolver defaults'], 'NewtonSolver()')
    assert s == dict(atol=1e-50, rtol=1e-30, max_it=3, error_on_nonconvergence=False)
    o = _engine_newton_opts('Newton')
    assert (o['kind'], o['atol'], o['rtol'], o['max_it']) == (0, s['atol'], s['rtol'], s['max_it'])
    from oracle.solvers import StatePath
    d = {k: v.default for k, v in inspect.signature(StatePath.solve_newton).parameters.items()}
    assert (d['atol'], d['rtol'], d['max_it']) == (s['atol'], s['rtol'], s['max_it'])
    init = _calls(ref['NewtonSolver(initialize=True)'], '__enter__.set')
    assert [e[2] for e in init] == [[0.1]] and not _calls(ref['NewtonSolver defaults'], '__enter__.set')


def test_snes_constants(ref):
    """utils_dolfinx.py:376-416 as executed: newtonls with the basic (full-step) line search, atol = rtol = 1e-13, max_it 100,
    error_on_nonconvergence, KSP preonly + LU (MUMPS) -- the direct solve the engine's Krylov methods replace."""
    ev = ref['SNESSolver']
    opts = {e[2]: e[3] for e in ev if e[0] == 'setitem'}
    assert opts == dict(snes_type='newtonls', snes_linesearch_type='basic', error_on_nonconvergence=True)
    (tol,) = [e[3] for e in _calls(ev, 'create().setTolerances')]
    assert tol == dict(atol=1e-13, rtol=1e-13, max_it=100)
    assert [e[2] for e in _calls(ev, 'getKSP().setType')] == [['preonly']] and [e[2] for e in _calls(ev, 'getPC().setType')] == [['lu']]
    o = _engine_newton_opts('SNES')
    assert (o['kind'], o['atol'], o['rtol'], o['max_it']) == (1, tol['atol'], tol['rtol'], tol['max_it'])
    assert o['stol'] == 1e-8                 # PETSc's default, which the reference leaves in force [upstream]
    from oracle.solvers import StatePath
    d = {k: v.default for k, v in inspect.signature(StatePath.solve_snes).parameters.items()}
    assert (d['atol'], d['rtol'], d['max_it'], d['stol']) == (tol['atol'], tol['rtol'], tol['max_it'], 1e-8)
    # solveNonlinear('SNES') solves in place on the state vector and reports the converged reason
    ev = ref['solveNonlinear SNES']
    assert [e[2] for e in _calls(ev, 'create().solve')] == [[None, '<w.vector>']] and _calls(ev, 'getConvergedReason')


def test_residual_lifting_convention(ref):
    """NonlinearSNESProblem.F (utils_dolfinx.py:352-367) as executed: apply_lifting(b, [a], bcs=[bcs], x0=[x], scale=-1),
    set_bc(b, bcs, x, -1), Jacobian assembled WITH the bcs.  The oracle's Newton residual must call its lifting the same way."""
    (lift,) = _calls(ref['NonlinearSNESProblem.F'], 'apply_lifting')
    (sbc,) = _calls(ref['NonlinearSNESProblem.F'], 'set_bc')
    assert lift[3] == dict(bcs=['<bcs>'], scale=-1.0, x0=['<x>']) and sbc[2] == ['<b>', '<bcs>', '<x>', -1.0]
    (jac,) = _calls(ref['NonlinearSNESProblem.J'], 'assemble_matrix')
    assert jac[3] == dict(bcs='<bcs>')
    from oracle import mesh as om, families as fam, assembly as asm, solvers
    from _cases import square_boundary_lists
    m = om.unit_square_tri(3)
    F = fam.PoissonP1(m)
    bc = asm.DirichletBC(F.N, square_boundary_lists(m.coords), 0.25)
    sp = solvers.StatePath(F, bc)
    seen = []
    real_lift, real_set, real_mat = asm.apply_lifting, asm.set_bc, asm.assemble_matrix
    asm.apply_lifting = lambda b, blocks, bc_, x0=None, scale=1.0: (seen.append(('lift', x0, scale)), real_lift(b, blocks, bc_, x0, scale))[1]
    asm.set_bc = lambda b, bc_, x0=None, scale=1.0: (seen.append(('set', x0, scale)), real_set(b, bc_, x0, scale))[1]
    asm.assemble_matrix = lambda blocks, shape, bc_=None: (seen.append(('mat', bc_)), real_mat(blocks, shape, bc_))[1]
    try:
        x = np.linspace(0.0, 1.0, F.N)
        sp.newton_F(x, [np.ones(F.M)])
        sp.newton_J(x, [np.ones(F.M)])
    finally:
        asm.apply_lifting, asm.set_bc, asm.assemble_matrix = real_lift, real_set, real_mat
    assert [s[0] for s in seen] == ['lift', 'set', 'mat']
    assert seen[0][1] is x and seen[0][2] == lift[3]['scale'] and seen[1][1] is x and seen[1][2] == sbc[2][3]
    assert seen[2][1] is bc


def test_system_assembly_convention(ref):
    """assembleSystem (utils_dolfinx.py:189-202) as executed: matrix with the bcs, right-hand side lifted with the DEFAULT
    x0 = None / scale = 1 and set_bc(b, bcs); assembleMatrix passes bcs=[] (no BC treatment: dR/du, dR/dm)."""
    ev = ref['assembleSystem']
    assert _calls(ev, 'assemble_matrix')[0][3] == dict(bcs='<bcs>')
    (lift,) = _calls(ev, 'apply_lifting')
    (sbc,) = _calls(ev, 'set_bc')
    assert len(lift[2]) == 3 and lift[3] == {} and len(sbc[2]) == 2 and sbc[3] == {}
    assert _calls(ref['assembleMatrix'], 'assemble_matrix')[0][3] == dict(bcs=[])
    from femo_b200.fea import utils_b200
    assert 'x0=None, scale=1' in utils_b200.assembleSystem.__doc__


def test_update_and_assemble_conventions(ref):
    """`update` broadcasts a length-1 array through Vec.set and copies anything else (quirk B6); `assemble` RETURNS a TypeError
    for an invalid dim (quirk B7).  The mirrors behave the same on the host."""
    assert [e[1] for e in ref['update length 1']] == ['v.vector.set']
    assert [e[0] for e in ref['update array']][0] == 'setitem'
    assert ref['assemble bad dim:result'] == 'TypeError'
    from femo_b200.fea import utils_b200 as ub, fem
    from femo_b200.fea.utils_b200 import createUnitSquareMesh
    mesh = createUnitSquareMesh(2)
    f = fem.Function(fem.FunctionSpace(mesh, ('DG', 0)))
    ub.update(f, np.array([2.5]))
    assert np.all(ub.getFuncArray(f) == 2.5)
    vals = np.arange(f.function_space.dim, dtype=np.float64)
    ub.update(f, vals)
    assert np.array_equal(ub.getFuncArray(f), vals)
    r = ub.assemble(None, dim=3)
    assert isinstance(r, TypeError)


def test_direct_solves_are_what_the_krylov_methods_replace(ref):
    """Every linear solve of the path is KSP preonly + LU(MUMPS) in the reference (exact up to round-off); the product's Krylov
    tolerance therefore sits well below every comparison tolerance of the parity tests."""
    for k in ('solveKSP_mumps', 'setUpKSP_MUMPS'):
        ev = ref[k]
        assert [e[2] for e in _calls(ev, 'create().setType')] == [['preonly']]
        assert [e[2] for e in _calls(ev, 'getPC().setType')] == [['lu']] and [e[2] for e in _calls(ev, 'setFactorSolverType')] == [['mumps']]
    assert [e[2] for e in _calls(ref['solveKSP_mumps'], 'create().solve')] == [['<b>', '<x>']]
    from femo_b200.fea.utils_b200 import KRYLOV
    assert KRYLOV['rtol'] <= 1e-10


def test_measures_projection_and_constants(ref):
    (meas,) = _calls(ref['createCustomMeasure ds'], 'ufl.Measure')
    assert meas[3]['metadata'] == dict(quadrature_degree=4)
    src = inspect.getsource(__import__('femo_b200.fea.utils_b200', fromlist=['x']).createCustomMeasure)
    assert '"quadrature_degree": 4' in src
    assert _calls(ref['project lumped'], 'pointwiseDivide') and not _calls(ref['project lumped'], 'KSP')
    assert _calls(ref['project'], 'KSP().create().solve')
    assert ref['DOLFIN_EPS'] == 3e-16
    from oracle import motor
    assert motor.DOLFIN_EPS == ref['DOLFIN_EPS']


LOCATE_GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'locate_dofs_reference.npz')


def _locate_inputs():
    """Seeded vertex cloud of an annulus band and query points near 11 of its vertices (polar and cartesian)."""
    rng = np.random.default_rng(4)
    th, r = rng.uniform(0, 2 * np.pi, 40), rng.uniform(0.06, 0.12, 40)
    nodes = np.stack([r * np.cos(th), r * np.sin(th), np.zeros(40)], axis=1)
    pick = rng.choice(40, 11, replace=False)
    polar = np.stack([th[pick], r[pick]], axis=1) + rng.normal(0, 1e-4, (11, 2))
    cart = nodes[pick, :2] + rng.normal(0, 1e-5, (11, 2))
    return nodes, pick, polar, cart


def test_locate_dofs_equals_the_recorded_reference_output():
    """locateDOFs / findNodeIndices of the mirror against what the reference's own functions return on the inputs of
    _locate_inputs(), stored in tests/golden/locate_dofs_reference.npz (held to a live reference run below)."""
    import types
    from femo_b200.fea import utils_b200 as ub
    z = np.load(LOCATE_GOLD)
    V = types.SimpleNamespace(tabulate_dof_coordinates=lambda: z['nodes'])
    polar = z['polar'].ravel().copy()
    assert np.array_equal(ub.locateDOFs(polar, V, input='polar'), z['polar_dofs'])
    assert np.array_equal(polar, z['polar'].ravel())                        # the mirror leaves its argument alone
    assert np.array_equal(ub.locateDOFs(z['cart'].copy(), V, input='cartesian'), z['cart_dofs'])
    assert np.array_equal(ub.findNodeIndices(z['cart'], z['nodes'][:, :2]), z['node_indices'])


def test_locate_dofs_equals_the_reference_function():
    """locateDOFs / findNodeIndices (utils_dolfinx.py:126-134,617-641) are plain numpy + KDTree code: the reference's own
    functions are CALLED here (polar and cartesian input) and must return the stored indices and the mirror's.  The reference
    converts the caller's array to cartesian IN PLACE as a side effect; the mirror leaves its argument alone."""
    if not L.REFERENCE or not os.path.isdir(os.path.join(L.REFERENCE, 'femo')):
        pytest.skip('no reference checkout')
    import types
    ref = L.load_reference_utils([])
    from femo_b200.fea import utils_b200 as ub
    nodes, pick, polar, cart = _locate_inputs()
    z = np.load(LOCATE_GOLD)
    assert all(np.array_equal(a, z[k]) for a, k in ((nodes, 'nodes'), (polar, 'polar'), (cart, 'cart')))
    V = types.SimpleNamespace(tabulate_dof_coordinates=lambda: nodes)
    a0, b0 = polar.ravel().copy(), polar.ravel().copy()
    ia, ib = ref.locateDOFs(a0, V, input='polar'), ub.locateDOFs(b0, V, input='polar')
    assert np.array_equal(ia, ib) and np.array_equal(ib[0::2] // 2, pick) and np.array_equal(ia, z['polar_dofs'])
    assert not np.array_equal(a0, polar.ravel()) and np.array_equal(b0, polar.ravel())
    ic = ref.locateDOFs(cart.copy(), V, input='cartesian')
    assert np.array_equal(ic, ub.locateDOFs(cart.copy(), V, input='cartesian')) and np.array_equal(ic, z['cart_dofs'])
    ni = ref.findNodeIndices(cart, nodes[:, :2])
    assert np.array_equal(ni, ub.findNodeIndices(cart, nodes[:, :2])) and np.array_equal(ni, z['node_indices'])
