"""The reference's OWN form code, executed: `pdeRes`, `outputForm`, `compliance`, `volume`, `averageFunc` ... are lifted out of
the example scripts under $FEMO_REFERENCE/examples (tests/_ufl_sympy.py: `ast` + a sympy implementation of the UFL operators
they use) and evaluated cell by cell on the meshes of the exact-integral fixtures.  The global residuals / functionals that come
out -- and their `sympy.diff` derivatives -- must equal tests/golden/symbolic/*.npz, i.e. the values the oracle (1e-13) and the
CUDA kernels (1e-12, tests/test_gpu_exact.py) are held to.  This closes the last hand-typed link: the fixtures are what the
reference's code says, integrated exactly.  Needs a reference checkout named by $FEMO_REFERENCE (skips without one); no GPU."""
import os

import numpy as np
import pytest

sp = pytest.importorskip('sympy')

import _ufl_sympy as U   # noqa: E402

REF_ROOT = os.path.abspath(os.environ['FEMO_REFERENCE']) if os.environ.get('FEMO_REFERENCE') else ''
REF = os.path.join(REF_ROOT, 'examples')
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'symbolic')
needs_reference = pytest.mark.skipif(not REF_ROOT or not os.path.isdir(REF), reason='no reference checkout')
# the fixture files the tests below were last run against: regenerating a fixture (scripts/make_symbolic_golden.py)
# fails test_fixtures_are_the_ones_checked_against_the_reference until these tests pass on it and its digest is updated
CHECKED = {
    'eb_beam.npz': '57461ae379fd5b731ce75b40d3a3e27f1cced7af7acf1fd2d10244e0adc9fdf7',
    'motor_em.npz': 'c9ebc38a13e814bea86d07857a352af0b1eaac6c6dda9be7d3d83fdf0244fafd',
    'motor_mm.npz': 'a54c5d2a880b8c953b6bdd28d5d5b334218e88b70b840fe24c888c2812f3be2f',
    'nlpoisson_p1.npz': 'fdff29f27d6dc280950910808c6d69f18ef1fc4c3818bf125f3143ae338911d5',
    'nlpoisson_p2.npz': '5d6c3fb3cf3d8dbffa695fa36fabeee5c45088ba30f2c17336e72b27161eac6a',
    'poisson_p1.npz': 'be53db5d94ad5916c3ec2c6ddd522b6812842a6f4109e858318118b33101cad6',
    'simp_hex8.npz': '0f112742358c8f8cf5ba2d0b5f40678e275e3c745fef398d6a59e4c3eb424208',
    'simp_q1.npz': '37a6b3b078f00e758fef7cb15b01e42505e76b4bdb1070be7fffd1f7bb024ffc',
}
TOL = 1e-13


@pytest.fixture(autouse=True)
def _reset_flags():
    U.POLYNOMIAL_COEFFICIENTS = True
    U.NUMERIC = {}
    yield
    U.POLYNOMIAL_COEFFICIENTS = True


def test_fixtures_are_the_ones_checked_against_the_reference():
    """tests/golden/symbolic/*.npz is written by the project's own sympy restatement (tests/test_oracle_symbolic.py); the tests
    below hold those fixtures to the reference's form code where a checkout is at hand.  Without one, the fixtures must still
    be the ones those tests passed on."""
    import hashlib
    for name, digest in CHECKED.items():
        with open(os.path.join(GOLD, name), 'rb') as f:
            assert hashlib.sha256(f.read()).hexdigest() == digest, name


def _num(exprs, tab):
    return np.array([float(sp.N(U.exactify(e).xreplace(tab), 30)) for e in exprs], dtype=np.float64)


def _same(got, exact, what):
    exact = np.asarray(exact, dtype=np.float64).reshape(np.shape(got))
    scale = max(np.abs(exact).max(), 1e-300)
    assert np.abs(np.asarray(got) - exact).max() <= TOL * scale, (what, np.abs(np.asarray(got) - exact).max() / scale)


def _compare(z, R, Js, Usym, Msym, tab):
    _same(_num(R, tab), z['R'], 'R')
    Rm = sp.Matrix([U.exactify(r) for r in R])
    _same(np.array(Rm.jacobian(list(Usym)).xreplace(tab).evalf(30), dtype=np.float64), z['A'], 'dR/du')
    _same(np.array(Rm.jacobian(list(Msym)).xreplace(tab).evalf(30), dtype=np.float64), z['D0'], 'dR/dm')
    for k, Jf in enumerate(Js):
        Jf = U.exactify(Jf)
        _same(_num([Jf], tab), z['J%d' % k], 'J%d' % k)
        _same(_num([sp.diff(Jf, s) for s in Usym], tab), z['Ju%d' % k], 'dJ%d/du' % k)
        _same(_num([sp.diff(Jf, s) for s in Msym], tab), z['Jm%d_0' % k], 'dJ%d/dm' % k)


def _table(z, Usym, Msym):
    tab = {Usym[i]: U.rat(z['state'][i]) for i in range(len(Usym))}
    tab.update({Msym[i]: U.rat(z['input0'][i]) for i in range(len(Msym))})
    return tab


def _tri_cells(z):
    """Cells of a triangle fixture with their exterior facets (edges that belong to one cell)."""
    cells = [tuple(int(v) for v in c) for c in z['cells']]
    X = [sp.Matrix([U.rat(a), U.rat(b)]) for a, b in z['coords']]
    cnt = {}
    for c in cells:
        for a in range(3):
            e = tuple(sorted((c[a], c[(a + 1) % 3])))
            cnt[e] = cnt.get(e, 0) + 1
    out = []
    for c in cells:
        ext = []
        for o in range(3):
            a, b = [k for k in range(3) if k != o]
            if cnt[tuple(sorted((c[a], c[b])))] == 1:
                ext.append(((a, b, o), None))
        out.append((c, U.Cell('triangle', [X[v] for v in c], ext)))
    return out, sorted(cnt)


@needs_reference
def test_poisson_forms_as_written_in_the_example():
    """examples/poisson_opt/run_poisson_opt.py: pdeRes(u, v, f) :136 (strong BCs are not part of the form), outputForm(u, f, u_ex) :115."""
    ns = U.load_defs(os.path.join(REF, 'poisson_opt', 'run_poisson_opt.py'))
    z = np.load(os.path.join(GOLD, 'poisson_p1.npz'))
    cells, _ = _tri_cells(z)
    N, M = z['state'].size, z['input0'].size
    Us, Fs = sp.symbols('U0:%d' % N), sp.symbols('F0:%d' % M)
    R, J = [0] * N, 0
    for c, (v, cell) in enumerate(cells):
        U.CTX = cell
        u = U.Field(sum(Us[v[a]] * cell.lam[a] for a in range(3)), coeffs=[Us[i] for i in v])
        uex = U.Field(sum(U.rat(z['meta_u_ex'][v[a]]) * cell.lam[a] for a in range(3)))
        f = U.Field(Fs[c])
        for a in range(3):
            test = U.Field(cell.lam[a], values=[1 if b == a else 0 for b in range(3)])
            R[v[a]] += ns['pdeRes'](u, test, f).value()
        J += ns['outputForm'](u, f, uex).value()
    _compare(z, R, [J], Us, Fs, _table(z, Us, Fs))


@pytest.mark.parametrize('degree', [1, 2])
@needs_reference
def test_nonlinear_poisson_forms_as_written_in_the_example(degree):
    """examples/nonlinear_poisson_opt/run_nonlinear_poisson_opt.py: pdeRes(u, v, f, u_exact=..., weak_bc=True, sym=True) :196-197,
    outputForm(u, f, u_ex) :172, with the fixture's polynomial u_exact (the example's sin field is not polynomial)."""
    ns = U.load_defs(os.path.join(REF, 'nonlinear_poisson_opt', 'run_nonlinear_poisson_opt.py'))
    z = np.load(os.path.join(GOLD, 'nlpoisson_p%d.npz' % degree))
    cells, edges = _tri_cells(z)
    nv = z['coords'].shape[0]
    eid = {e: k for k, e in enumerate(edges)}
    N, M = z['state'].size, z['input0'].size
    Us, Fs = sp.symbols('U0:%d' % N), sp.symbols('F0:%d' % M)
    R, J = [0] * N, 0
    for c, (v, cell) in enumerate(cells):
        U.CTX = cell
        lam = cell.lam
        if degree == 1:
            dofs, phi = list(v), lam
        else:
            dofs = list(v) + [nv + eid[tuple(sorted((v[(i + 1) % 3], v[(i + 2) % 3])))] for i in range(3)]
            phi = [l * (2 * l - 1) for l in lam] + [4 * lam[(i + 1) % 3] * lam[(i + 2) % 3] for i in range(3)]
        u = U.Field(sum(Us[d] * p for d, p in zip(dofs, phi)), coeffs=[Us[d] for d in dofs])
        x, y = cell.x
        uex = x * x * y - 3 * x * y + y ** 3 / 4 + sp.Rational(1, 2)
        f = U.Field(Fs[c])
        for a, d in enumerate(dofs):
            test = U.Field(phi[a], values=[1 if b == a else 0 for b in range(len(dofs))])
            R[d] += ns['pdeRes'](u, test, f, u_exact=uex, weak_bc=True, sym=True).value()
        J += ns['outputForm'](u, f, uex).value()
    _compare(z, R, [J], Us, Fs, _table(z, Us, Fs))


@needs_reference
def test_beam_forms_as_written_in_the_example():
    """examples/beam_thickness_opt/run_thickness_opt_cantilever_beam.py: pdeRes(u, v, t, f, ds_(100), E, width) :127-131,
    compliance(u, f, ds_(100)) :135, volume(t, width, L) :137; Hermite-3 with reference-derivative slope dofs."""
    ns = U.load_defs(os.path.join(REF, 'beam_thickness_opt', 'run_thickness_opt_cantilever_beam.py'))
    z = np.load(os.path.join(GOLD, 'eb_beam.npz'))
    Eb, width, L, fload = (float(v) for v in z['meta_params'])
    xs = z['coords'][:, 0]
    nc = z['cells'].shape[0]
    N, M = z['state'].size, z['input0'].size
    Us, Ts = sp.symbols('U0:%d' % N), sp.symbols('T0:%d' % M)
    xi = sp.Symbol('xi_0')
    a_ = sp.symbols('a0:4')
    cubic = sum(a_[i] * xi ** i for i in range(4))
    conds = [cubic.subs(xi, 0), sp.diff(cubic, xi).subs(xi, 0), cubic.subs(xi, 1), sp.diff(cubic, xi).subs(xi, 1)]
    basis = [cubic.subs(sp.solve([conds[i] - (1 if i == k else 0) for i in range(4)], a_)) for k in range(4)]
    f = U.Constant(None, fload)
    ds100 = U.NAMESPACE['ds'](100)
    R, comp, vol = [0] * N, 0, 0
    for c in range(nc):
        ext = [((0, 1), 100)] if c == nc - 1 else ([((0, 0), 0)] if c == 0 else [])
        U.CTX = U.Cell('interval', [sp.Matrix([U.rat(xs[c])]), sp.Matrix([U.rat(xs[c + 1])])], ext)
        dofs = [2 * c, 2 * c + 1, 2 * c + 2, 2 * c + 3]
        u = U.Field(sum(Us[d] * p for d, p in zip(dofs, basis)), coeffs=[Us[d] for d in dofs])
        t = U.Field(Ts[c])
        for a, d in enumerate(dofs):
            test = U.Field(basis[a], values=[1 if b == a else 0 for b in range(4)])
            R[d] += ns['pdeRes'](u, test, t, f, ds100, Eb, width).value()
        comp += ns['compliance'](u, f, ds100).value()
        vol += ns['volume'](t, width, L).value()
    _compare(z, R, [comp, vol], Us, Ts, _table(z, Us, Ts))


@pytest.mark.parametrize('name', ['simp_q1', 'simp_hex8'])
@needs_reference
def test_simp_forms_as_written_in_the_example(name):
    """examples/beam_topo_opt/run_topo_opt_cantilever_beam.py: pdeRes(u, v, rho, f, dss=ds_(100), method='SIMP') :102-107,
    averageFunc(rho) :111, compliance(u, f, dss=ds_(100)) :113-115.  The form is written for any dimension (`len(u)`,
    `Identity(d)`), so the same reference code defines the 3-D hexahedral extension."""
    z = np.load(os.path.join(GOLD, name + '.npz'))
    d = z['coords'].shape[1]
    prm = [float(v) for v in z['meta_params']]
    assert prm[0] == 0.3 and prm[-1] == 3.0                     # the script hard-codes nu = 0.3 and the cubic SIMP law
    cells = z['cells']
    X = z['coords']
    lo, hi = X.min(axis=0), X.max(axis=0)
    total = float(np.prod(hi - lo))
    ns = U.load_defs(os.path.join(REF, 'beam_topo_opt', 'run_topo_opt_cantilever_beam.py'),
                     extra=dict(mesh=None, assemble=lambda form: U.rat(total), Function=lambda V: U.Field(sp.Integer(0))))
    N, M = z['state'].size, z['input0'].size
    Us, Rs = sp.symbols('U0:%d' % N), sp.symbols('R0:%d' % M)
    fvec = U.Constant(None, tuple(prm[1:1 + d]))
    ds100 = U.NAMESPACE['ds'](100)
    R, avg, comp = [0] * N, 0, 0
    for c, verts in enumerate(cells):
        Xc = [sp.Matrix([U.rat(v) for v in X[k]]) for k in verts]
        ext = []
        for k in range(d):
            if X[verts[0]][k] == lo[k]:
                ext.append(((k, 0), 0))
            if X[verts[-1]][k] == hi[k]:
                ext.append(((k, 1), 100 if k == 0 else 0))          # the traction faces of the fixture: x = x_max
        cell = U.CTX = U.Cell('box', Xc, ext)
        phi = [sp.Mul(*[(cell.xi[k] if (a >> k) & 1 else 1 - cell.xi[k]) for k in range(d)]) for a in range(2 ** d)]
        dofs = [[int(verts[a]) * d + k for k in range(d)] for a in range(2 ** d)]
        flat = [dofs[a][k] for a in range(2 ** d) for k in range(d)]
        u = U.Field(sp.Matrix([sum(Us[dofs[a][k]] * phi[a] for a in range(2 ** d)) for k in range(d)]), coeffs=[Us[i] for i in flat])
        rho = U.Field(Rs[c])
        for a in range(2 ** d):
            for k in range(d):
                test = U.Field(sp.Matrix([phi[a] if i == k else 0 for i in range(d)]))
                R[dofs[a][k]] += ns['pdeRes'](u, test, rho, fvec, dss=ds100, method='SIMP').value()
        avg += ns['averageFunc'](rho).value()
        comp += ns['compliance'](u, fvec, dss=ds100).value()
    _compare(z, R, [avg, comp], Us, Rs, _table(z, Us, Rs))


# ------------------------------------------------------------------------------------------------- config 5 (motor)
def _motor_namespace():
    """examples/em_motor_opt/motor_pde.py with what it star-imports: the ALE kinematics gradx / J / F and DOLFIN_EPS from
    femo/fea/utils_dolfinx.py:30-66 (the reference's own definitions, executed), and the B-H curve pieces of
    permeability/piecewise_permeability.py fed with the fitted constants of femo_b200/forms/bh_fit.json (that module fits them
    from a data table at import time)."""
    import json
    fit = json.load(open(os.path.join(os.path.dirname(GOLD), '..', '..', 'femo_b200', 'forms', 'bh_fit.json')))
    utils = U.load_defs(os.path.join(REF_ROOT, 'femo', 'fea', 'utils_dolfinx.py'))
    perm = U.load_defs(os.path.join(REF, 'em_motor_opt', 'permeability', 'piecewise_permeability.py'),
                       extra=dict(linearA=fit['lin'][0], linearB=fit['lin'][1], cubicA=fit['cubic'][0], cubicB=fit['cubic'][1],
                                  cubicC=fit['cubic'][2], cubicD=fit['cubic'][3], popt_exp=fit['exp'], x1=fit['x1'], x2=fit['x2']))
    extra = {k: utils[k] for k in ('gradx', 'J', 'F', 'DOLFIN_EPS')}
    extra.update({k: perm[k] for k in ('linearPortion', 'cubicPortion')})
    extra.update(exp_coeff=perm['extractexpDecayCoeff'](), cubic_bounds=perm['extractCubicBounds']())
    return U.load_defs(os.path.join(REF, 'em_motor_opt', 'motor_pde.py'), extra=extra)


def _motor_cells(z, tagged):
    """Triangle cells with their tagged facets: `tagged` = set of (cell, local facet) pairs (local facet i is opposite local
    vertex i) carrying tag 1000, or None for every exterior facet untagged (`ds` without a subdomain id)."""
    cells = [tuple(int(v) for v in c) for c in z['cells']]
    X = [sp.Matrix([U.rat(a), U.rat(b)]) for a, b in z['coords']]
    cnt = {}
    for c in cells:
        for a in range(3):
            e = tuple(sorted((c[a], c[(a + 1) % 3])))
            cnt[e] = cnt.get(e, 0) + 1
    tags = z['meta_cell_tags']
    out = []
    for ci, c in enumerate(cells):
        ext, inner = [], []
        for o in range(3):
            a, b = [k for k in range(3) if k != o]
            boundary = cnt[tuple(sorted((c[a], c[b])))] == 1
            if tagged is None:
                if boundary:
                    ext.append(((a, b, o), None))
            elif (ci, o) in tagged:
                (ext if boundary else inner).append(((a, b, o), 1000))
        out.append((c, U.Cell('triangle', [X[v] for v in c], ext, cell_tag=int(tags[ci]), interior=inner)))
    return out


MESH2D = __import__('types').SimpleNamespace(topology=__import__('types').SimpleNamespace(dim=2))


def _vector_p1(cell, v, syms):
    coeffs = [syms[2 * v[a] + k] for a in range(3) for k in range(2)]
    return U.Field(sp.Matrix([sum(syms[2 * v[a] + k] * cell.lam[a] for a in range(3)) for k in range(2)]), coeffs=coeffs, mesh=MESH2D)


def _compare_numeric(z, R, Js, Usym, Msym, tab, tol):
    def same(got, exact, what):
        exact = np.asarray(exact, dtype=np.float64).reshape(np.shape(got))
        scale = max(np.abs(exact).max(), 1e-300)
        assert np.abs(np.asarray(got) - exact).max() <= tol * scale, (what, np.abs(np.asarray(got) - exact).max() / scale)
    same(_num(R, tab), z['R'], 'R')
    same(U.jac_numeric(R, Usym, tab), z['A'], 'dR/du')
    same(U.jac_numeric(R, Msym, tab), z['D0'], 'dR/dm')
    for k, Jf in enumerate(Js):
        same(_num([Jf], tab), z['J%d' % k], 'J%d' % k)
        same(U.jac_numeric([Jf], Usym, tab)[0], z['Ju%d' % k], 'dJ%d/du' % k)
        same(U.jac_numeric([Jf], Msym, tab)[0], z['Jm%d_0' % k], 'dJ%d/dm' % k)


@needs_reference
def test_mesh_motion_forms_as_written_in_the_example():
    """motor_pde.pdeResMM(uhat, v, g=..., nitsche=True, sym=True, overpenalty=False, dS_=dS(1000), ds_=ds(1000)) and
    area_form(uhat, dx, ids) as run_motor_opt.py:176-187 calls them; `X("+")` restrictions are rewritten to restricted(X, "+")."""
    ns = _motor_namespace()
    z = np.load(os.path.join(GOLD, 'motor_mm.npz'))
    tagged = {(int(c), int(l)) for c, l in zip(z['meta_facet_cells'], z['meta_facet_locals'])}
    cells = _motor_cells(z, tagged)
    N = z['state'].size
    Us, Gs = sp.symbols('U0:%d' % N), sp.symbols('G0:%d' % N)
    tab = _table(z, Us, Gs)
    U.NUMERIC = tab
    U.POLYNOMIAL_COEFFICIENTS = False
    dx, dS, ds = U.NAMESPACE['dx'], U.NAMESPACE['dS'], U.NAMESPACE['ds']
    R, areas = [0] * N, [0, 0, 0]
    for v, cell in cells:
        U.CTX = cell
        uhat, g = _vector_p1(cell, v, Us), _vector_p1(cell, v, Gs)
        for a in range(3):
            for k in range(2):
                test = U.Field(sp.Matrix([cell.lam[a] if i == k else 0 for i in range(2)]),
                               values=[1 if (b, j) == (a, k) else 0 for b in range(3) for j in range(2)], mesh=MESH2D)
                R[2 * v[a] + k] += ns['pdeResMM'](uhat, test, g=g, nitsche=True, sym=True, overpenalty=False,
                                                  dS_=dS(1000), ds_=ds(1000)).value()
        for k, ids in enumerate((15, 3, [1, 2])):                       # winding_id, magnet_id, steel_id (run_motor_opt.py:68-70)
            areas[k] += ns['area_form'](uhat, dx, ids).value()
    _compare_numeric(z, R, areas, Us, Gs, tab, 1e-12)


@needs_reference
def test_magnetostatics_forms_as_written_in_the_example():
    """motor_pde.pdeResEM(u, v, uhat, iq, dx, p, s, Hc, vacuum_perm, angle, g=0, nitsche=True, sym=True, overpenalty=False, ds_=ds)
    and B_power_form(u, uhat, n, dx, [1, 2]) as run_motor_opt.py:276-291 calls them -- RelativePermeability, JS, the 216
    subdomain integrals and the Nanson-normal Nitsche terms all come from the reference's code."""
    ns = _motor_namespace()
    z = np.load(os.path.join(GOLD, 'motor_em.npz'))
    cells = _motor_cells(z, None)
    N, M = z['state'].size, z['input0'].size
    Us, Ws = sp.symbols('U0:%d' % N), sp.symbols('W0:%d' % M)
    tab = _table(z, Us, Ws)
    U.NUMERIC = tab
    U.POLYNOMIAL_COEFFICIENTS = False
    dx, ds = U.NAMESPACE['dx'], U.NAMESPACE['ds']
    prm = {k: float(z['meta_' + k]) for k in ('Hc', 'angle', 'iq')}
    p_, s_ = int(z['meta_p']), int(z['meta_s'])
    assert float(z['meta_beta']) == 1e4                               # hard-coded in pdeResEM
    mu0 = 4e-7 * np.pi
    R, outs = [0] * N, [0, 0]
    for v, cell in cells:
        U.CTX = cell
        u = U.Field(sum(Us[v[a]] * cell.lam[a] for a in range(3)), coeffs=[Us[i] for i in v], mesh=MESH2D)
        uhat = _vector_p1(cell, v, Ws)
        zero = U.Field(sp.Integer(0), mesh=MESH2D)
        for a in range(3):
            test = U.Field(cell.lam[a], values=[1 if b == a else 0 for b in range(3)], mesh=MESH2D)
            R[v[a]] += ns['pdeResEM'](u, test, uhat, prm['iq'], dx, p_, s_, prm['Hc'], mu0, prm['angle'],
                                      g=zero, nitsche=True, sym=True, overpenalty=False, ds_=ds).value()
        for k, n_ in enumerate((2, 1.76835)):
            outs[k] += ns['B_power_form'](u, uhat, n_, dx, [1, 2]).value()
    _compare_numeric(z, R, outs, Us, Ws, tab, 1e-11)
