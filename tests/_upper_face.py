"""Differential harness for the UPPER face of the drop-in boundary (SURVEY.md section 8b): the reference's own Python layer
-- `FEA` (femo/fea/fea_dolfinx.py:70-234), `StateOperation`, `OutputOperation`, `OutputFieldOperation`, `FEAModel`
(femo/csdl_opt/*.py) -- imported UNMODIFIED from a reference checkout and run over a recording stub of everything below
it (dolfinx / ufl / PETSc and femo's utils_dolfinx functions), against femo_b200's mirrors run over the SAME stub.

The stub lower face returns deterministic vectors that depend on what it was called with, so both the sequence of
lower-face calls (names, arguments) and every value a callback writes into the CSDL containers can be compared exactly.
Nothing here touches the GPU engine or oracle/: it is about who calls what, in which order, with which arrays, and
assign-versus-accumulate semantics.  scripts/make_upper_face_trace.py stores the reference's run as
tests/golden/upper_face_trace.json (the reference cannot travel to the GPU box); tests/test_upper_face.py compares the
mirrors with it and, where $FEMO_REFERENCE names a reference checkout, regenerates it live.
"""
import importlib
import importlib.util
import os
import sys
import types
import zlib

import numpy as np

# a checkout of the reference femo project; what runs its code skips without one
REFERENCE = os.path.abspath(os.environ['FEMO_REFERENCE']) if os.environ.get('FEMO_REFERENCE') else ''


def vec(key, n):
    """Deterministic pseudo-data keyed by a description of the call."""
    return np.sin((zlib.crc32(key.encode()) % 9973) + 1.25 * np.arange(n))


def digest(a):
    a = np.ravel(np.asarray(a, dtype=np.float64))
    return repr(float(a @ np.cos(np.arange(1, a.size + 1)))) + '/%d' % a.size


class World:
    """One recording stub world: the names a module body imports from femo.fea.fea_dolfinx / utils_dolfinx / dolfinx / ufl."""

    def __init__(self):
        self.events = []
        w = self

        class Space:
            num_sub_spaces = 0

            def __init__(self, n, name='V'):
                self.n, self.name = n, name

        class Vec:
            def __init__(self, f):
                self.f = f

            def set(self, v):
                w.log('Vec.set', self.f.name, float(v))
                self.f.values[:] = v

            def getArray(self):
                w.log('Vec.getArray', self.f.name)
                return self.f.values

            array = property(lambda self: self.f.values)

            def assemble(self):
                pass

            def ghostUpdate(self, *a, **k):
                pass

        class XView:
            def __init__(self, f):
                self.f = f

            @property
            def array(self):
                return self.f.values

        class Function:
            count = 0

            def __init__(self, V, name=None):
                Function.count += 1
                self.function_space = V
                self.name = name or 'w%d' % Function.count
                self.values = np.zeros(V.n)
                self.vector = Vec(self)
                self.x = XView(self)

            def rename(self, a, b=None):
                self.name = a

        class Form:
            def __init__(self, text, size=None):
                self.text, self.size = text, size

        class Mat:
            def __init__(self, text, plain=None):
                self.text = text
                if plain is not None:
                    self.plain = plain

        class Ksp:
            def __init__(self, A):
                self.A = A

            def solve(self, b, x):
                w.log('ksp.solve', self.A.text, b.f.name, digest(b.f.values), x.f.name)
                x.f.values[:] = vec('ksp|%s|%s' % (self.A.text, digest(b.f.values)), x.f.values.size)

        class Recorder:
            def __init__(self, *a, **k):
                w.log('recorder.open')

            def write_mesh(self, mesh):
                w.log('recorder.write_mesh')

            def write_function(self, f, t=0):
                w.log('recorder.write_function', f.name, int(t))

        self.Space, self.Function, self.Form, self.Mat, self.Recorder = Space, Function, Form, Mat, Recorder

        def state_key():
            return '|'.join('%s=%s' % (f.name, digest(f.values)) for f in self.tracked)

        def update(f, a):
            a = np.asarray(a, dtype=np.float64)
            self.log('update', f.name, digest(a))
            f.values[:] = a if a.size != 1 else float(a.ravel()[0])

        def setFuncArray(f, a):
            self.log('setFuncArray', f.name, digest(a))
            f.values[:] = np.asarray(a, dtype=np.float64)

        def getFuncArray(f):
            self.log('getFuncArray', f.name)
            return f.values

        def getFormArray(form):
            return np.zeros(form.size)

        def assembleVector(form):
            self.log('assembleVector', form.text)
            return vec('V|%s|%s' % (form.text, state_key()), form.size)

        def assembleMatrix(form, bcs=[]):
            self.log('assembleMatrix', form.text, len(bcs))
            return Mat('M[%s]' % form.text)

        def assembleSystem(J, F, bcs=[], rhs=True):
            self.log('assembleSystem', J.text, F.text, len(bcs))
            return Mat('A[%s|%d]' % (J.text, len(bcs)), plain=Mat('M[%s]' % J.text)), vec('b|' + F.text, F.size)

        def computePartials(form, func):
            self.log('computePartials', form.text, func.name)
            return Form('d(%s)/d(%s)' % (form.text, func.name), func.values.size)

        def derivative(form, func, *a):
            return Form('d(%s)/d(%s)' % (form.text, func.name), func.values.size)

        def createFunction(func):
            self.log('createFunction', func.name)
            g = Function(func.function_space, 'copy(%s)' % func.name)
            g.values[:] = func.values
            return g

        def mv(kind, A, x, n):
            self.log(kind, A.text, x.name, digest(x.values))
            return vec('%s|%s|%s' % (kind, A.text, digest(x.values)), n)

        def computeMatVecProductFwd(A, x):
            return mv('computeMatVecProductFwd', A, x, self.rows[A.text])

        def computeMatVecProductBwd(A, R):
            return mv('computeMatVecProductBwd', A, R, self.cols[A.text])

        def setUpKSP_MUMPS(A):
            self.log('setUpKSP_MUMPS', A.text)
            return Ksp(A)

        def transpose(A):
            return Mat('T(%s)' % A.text)

        def solveKSP_mumps(A, b, x):
            self.log('solveKSP_mumps', A.text, b.f.name, digest(b.f.values), x.f.name)
            x.f.values[:] = vec('solve|%s|%s' % (A.text, digest(b.f.values)), x.f.values.size)

        def assemble(form, dim=0, bcs=[]):
            self.log('assemble', form.text, dim)
            if dim == 0:
                return float(vec('s|%s|%s' % (form.text, state_key()), 1)[0])
            return vec('a|%s|%s' % (form.text, state_key()), form.size)

        def solveNonlinear(res, func, bc, solver, report, initialize):
            self.log('solveNonlinear', res.text, func.name, len(bc), solver, bool(report), bool(initialize))
            func.values[:] = vec('state|%s|%s' % (res.text, state_key()), func.values.size)

        def project(form, func, lump_mass=False):
            self.log('project', form.text, func.name, bool(lump_mass))
            func.values[:] = vec('proj|%s|%s' % (form.text, state_key()), func.values.size)

        def FunctionSpace(mesh, element):
            return Space(5, 'CG1(out)')

        def dirichletbc(ubc, dofs, V=None):
            self.log('dirichletbc', str(ubc), list(dofs), V is not None)
            return ('bc', str(ubc), tuple(dofs))

        mpi = types.SimpleNamespace(COMM_WORLD='comm')
        self.names = dict(update=update, setFuncArray=setFuncArray, getFuncArray=getFuncArray, getFormArray=getFormArray,
                          assembleVector=assembleVector, assembleMatrix=assembleMatrix, assembleSystem=assembleSystem,
                          computePartials=computePartials, derivative=derivative, createFunction=createFunction,
                          computeMatVecProductFwd=computeMatVecProductFwd, computeMatVecProductBwd=computeMatVecProductBwd,
                          setUpKSP_MUMPS=setUpKSP_MUMPS, transpose=transpose, solveKSP_mumps=solveKSP_mumps,
                          assemble=assemble, solveNonlinear=solveNonlinear, project=project, FunctionSpace=FunctionSpace,
                          Function=Function, dirichletbc=dirichletbc, XDMFFile=Recorder, NpyRecorder=Recorder, MPI=mpi)
        self.tracked = []
        self.rows, self.cols = {}, {}

    def log(self, *ev):
        self.events.append(list(ev))

    def take(self):
        ev, self.events = self.events, []
        return ev


# ---------------------------------------------------------------------------------------------------------------
def _csdl_module():
    from femo_b200.csdl_opt import _csdl_compat as cc
    m = types.ModuleType('csdl')
    m.Model, m.CustomImplicitOperation, m.CustomExplicitOperation = cc.Model, cc.CustomImplicitOperation, cc.CustomExplicitOperation
    m.custom = cc.csdl.custom
    return m


def load_reference(world, root=REFERENCE):
    """The reference's four modules, executed from their own files under stub imports."""
    stubs = {}

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        if '.' not in name or name in ('femo.fea', 'femo.csdl_opt', 'dolfinx.fem', 'matplotlib.pyplot'):
            m.__path__ = []
        stubs[name] = m
        return m
    n = world.names
    mod('femo')
    mod('femo.fea')
    mod('femo.csdl_opt')
    mod('femo.fea.utils_dolfinx', **n)
    mod('dolfinx')
    mod('dolfinx.io', XDMFFile=n['XDMFFile'])
    mod('dolfinx.fem', set_bc=None, Function=n['Function'], FunctionSpace=n['FunctionSpace'], dirichletbc=n['dirichletbc'],
        locate_dofs_topological=None, locate_dofs_geometrical=None, Constant=None, VectorFunctionSpace=None)
    mod('dolfinx.fem.petsc', apply_lifting=None)
    mod('ufl', grad=None, SpatialCoordinate=None, CellDiameter=None, FacetNormal=None, div=None, Identity=None)
    mod('matplotlib')
    mod('matplotlib.pyplot')
    stubs['csdl'] = _csdl_module()
    saved = {k: sys.modules.get(k) for k in stubs}
    sys.modules.update(stubs)
    try:
        def load(name, rel):
            spec = importlib.util.spec_from_file_location(name, os.path.join(root, rel))
            m = importlib.util.module_from_spec(spec)
            sys.modules[name] = m
            stubs[name] = m
            saved.setdefault(name, None)
            spec.loader.exec_module(m)
            return m
        fea = load('femo.fea.fea_dolfinx', 'femo/fea/fea_dolfinx.py')
        sm = load('femo.csdl_opt.state_model', 'femo/csdl_opt/state_model.py')
        om = load('femo.csdl_opt.output_model', 'femo/csdl_opt/output_model.py')
        fm = load('femo.csdl_opt.fea_model', 'femo/csdl_opt/fea_model.py')
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return dict(FEA=fea.FEA, StateOperation=sm.StateOperation, OutputOperation=om.OutputOperation,
                OutputFieldOperation=om.OutputFieldOperation, FEAModel=fm.FEAModel)


class patched:
    """femo_b200's mirrors with the stub world's names in place of their lower face (restored on exit)."""

    def __init__(self, world):
        self.world = world

    def __enter__(self):
        from femo_b200.fea import fea_b200
        from femo_b200.csdl_opt import state_model, output_model, fea_model
        self.saved = []
        for m in (fea_b200, state_model, output_model):
            for k, v in self.world.names.items():
                if k in m.__dict__:
                    self.saved.append((m, k, m.__dict__[k]))
                    m.__dict__[k] = v
        from femo_b200.fea import utils_b200
        self.saved.append((utils_b200, 'project', utils_b200.project))
        utils_b200.project = self.world.names['project']                 # FEA.projectFieldOutput imports it at call time
        return dict(FEA=fea_b200.FEA, StateOperation=state_model.StateOperation, OutputOperation=output_model.OutputOperation,
                    OutputFieldOperation=output_model.OutputFieldOperation, FEAModel=fea_model.FEAModel)

    def __exit__(self, *a):
        for m, k, v in reversed(self.saved):
            m.__dict__[k] = v


# ---------------------------------------------------------------------------------------------------------------
def _snap(d):
    return {str(k): (np.ravel(np.asarray(v, dtype=np.float64)).tolist()) for k, v in d.items()}


def scenario(world, impl):
    """A fixed script of registry calls and CSDL callbacks; returns [(step name, lower-face events, container values)]."""
    W = world
    out = []

    def step(name, **containers):
        out.append([name, W.take(), {k: _snap(v) for k, v in containers.items()}])

    NU, NF = 4, 6
    f = W.Function(W.Space(NF, 'DG0'), 'f0')
    u = W.Function(W.Space(NU, 'CG1'), 'u0')
    W.tracked = [u, f]
    R = W.Form('R(u,f)', NU)
    J = W.Form('J(u,f)')
    fea = impl['FEA']('mesh')
    f.values[:] = 7.0
    fea.add_input('f', f, init_val=0.5)                                   # overwrites the function (quirk B5)
    try:
        fea.add_input('f', f)
        dup = 'no error'
    except ValueError as e:
        dup = 'ValueError: %s' % e
    fea.add_state(name='u', function=u, residual_form=R, arguments=['f'])
    fea.add_output(name='J', type='scalar', form=J, arguments=['u', 'f'])
    fea.add_field_output('field', W.Form('F(u)', 5), ['u'])
    fea.add_strong_bc('ubc', [[0, 1], [3]])
    W.rows.update({'M[d(R(u,f))/d(u0)]': NU, 'M[d(R(u,f))/d(f0)]': NU})
    W.cols.update({'M[d(R(u,f))/d(u0)]': NU, 'M[d(R(u,f))/d(f0)]': NF})
    reg = dict(f_after_add_input=f.values.copy(),
               shapes=[fea.inputs_dict['f']['shape'], fea.states_dict['u']['shape'], fea.outputs_dict['J']['shape'],
                       fea.outputs_field_dict['field']['shape']], nbc=[len(fea.bc)],
               state_keys=[float(len(sorted(fea.states_dict['u'])))], flags=[float(fea.opt_iter), float(fea.linear_problem)])
    step('registry', reg=reg)
    reg_keys = dict(inputs=sorted(fea.inputs_dict['f']), states=sorted(fea.states_dict['u']), outputs=sorted(fea.outputs_dict['J']),
                    field=sorted(fea.outputs_field_dict['field']),
                    partials=[p.text for p in fea.outputs_dict['J']['partials']],
                    attrs=sorted(k for k in vars(fea) if not k.startswith('_')), duplicate_input=dup)
    out.append(['registry-keys', [], reg_keys])

    def state_op():
        return impl['StateOperation'](fea=fea, args_dict={'f': fea.inputs_dict['f']}, state_name='u', debug_mode=False)
    op = state_op()
    step('StateOperation.define', meta=dict(inputs=[float(s) for s in op.input_meta['f']['shape']],
                                            outputs=[float(s) for s in op.output_meta['u']['shape']]))
    fin, uin = vec('f-in', NF), vec('u-in', NU)
    res = {}
    op.evaluate_residuals({'f': fin}, {'u': uin}, res)
    step('evaluate_residuals', residuals=res)
    outs = {'u': uin.copy()}
    op.solve_residual_equations({'f': fin}, outs)
    step('solve_residual_equations', outputs=outs, opt_iter={'n': [fea.opt_iter]})
    calls = []
    fea.custom_solve = lambda r, fn, bc, report: calls.append((r.text, fn.name, len(bc), report))
    op.solve_residual_equations({'f': fin}, outs)
    op.solve_residual_equations({'f': fin}, outs)                         # sticky: initial_solve is never cleared (quirk B9)
    step('custom_solve twice', calls={'n': [len(calls)], 'initial_solve': [float(fea.initial_solve)]})
    fea.custom_solve = None
    op.compute_derivatives({'f': fin}, {'u': uin}, {})
    step('compute_derivatives', held=dict(dRdu=[0.0] if op.dRdu is not None else [], ksp=[] if op.ksp is None else [1.0]))
    for mode in ('fwd', 'rev'):
        d_in, d_out, d_res = {'f': vec('df', NF)}, {'u': vec('du', NU)}, {'u': vec('dr', NU)}
        op.compute_jacvec_product({'f': fin}, {'u': uin}, d_in, d_out, d_res, mode)
        step('compute_jacvec_product ' + mode, d_inputs=d_in, d_outputs=d_out, d_residuals=d_res)
        d_in, d_res = {}, {'u': vec('dr2', NU)}                             # containers that lack keys: nothing is touched
        op.compute_jacvec_product({'f': fin}, {'u': uin}, d_in, {}, d_res, mode)
        step('compute_jacvec_product %s, absent keys' % mode, d_inputs=d_in, d_residuals=d_res)
    for linear in (False, True):
        fea.linear_problem = linear
        op = state_op()
        op.compute_derivatives({'f': fin}, {'u': uin}, {})
        W.take()
        for mode in ('fwd', 'rev'):
            d_out, d_res = {'u': vec('seed-out', NU)}, {'u': vec('seed-res', NU)}
            op.apply_inverse_jacobian(d_out, d_res, mode)
            step('apply_inverse_jacobian %s linear=%s' % (mode, linear), d_outputs=d_out, d_residuals=d_res)
    fea.linear_problem = False
    oop = impl['OutputOperation'](fea=fea, args_dict={'u': fea.states_dict['u'], 'f': fea.inputs_dict['f']}, output_name='J')
    o = {}
    oop.compute({'u': uin, 'f': fin}, o)
    step('OutputOperation.compute', outputs=o)
    d = {}
    oop.compute_derivatives({'u': uin, 'f': fin}, d)
    step('OutputOperation.compute_derivatives', derivatives=d)
    fop = impl['OutputFieldOperation'](fea=fea, args_dict={'u': fea.states_dict['u']}, output_name='field')
    o = {}
    fop.compute({'u': uin}, o)
    step('OutputFieldOperation.compute', outputs=o)
    # the whole chain through FEAModel and the backend stand-in: run() then reverse-mode totals
    import contextlib
    import io
    from femo_b200.csdl_opt._csdl_compat import Simulator
    with contextlib.redirect_stdout(io.StringIO()):                       # FEAModel switches debug_mode on (fea_model.py:15)
        sim = Simulator(impl['FEAModel'](fea=[fea]), pinned=False)
        W.take()
        sim['f'] = fin
        sim.run()
        step('FEAModel run', vars={k: np.asarray(v) for k, v in sim.vars.items()})
        tot = sim.compute_totals('J', 'f')
        step('FEAModel compute_totals', totals={'dJdf': tot[('J', 'f')]})
    return out
