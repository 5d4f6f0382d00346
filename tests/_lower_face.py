"""What femo itself asks dolfinx / PETSc to do on the hot path, recorded by running the reference's own
femo/fea/utils_dolfinx.py (imported unmodified from a reference checkout) over a recording stand-in for dolfinx, ufl, petsc4py
and mpi4py: solver types and tolerances, the lifting / set_bc conventions of the Newton and SNES residuals, the BC'd system
assembly, `update`'s broadcast, `assemble`'s error convention, the quadrature degree of custom measures.  These are the facts the
oracle (oracle/solvers.py, oracle/assembly.py) and the engine's defaults restate; tests/test_lower_face.py compares them with
the recording committed as tests/golden/lower_face_calls.json (scripts/make_lower_face_calls.py)."""
import importlib.util
import os
import sys
import types

import numpy as np

# a checkout of the reference femo project; what runs its code skips without one
REFERENCE = os.path.abspath(os.environ['FEMO_REFERENCE']) if os.environ.get('FEMO_REFERENCE') else ''


class Rec:
    """Records every call / attribute assignment / item assignment made on it or on anything reached from it."""

    def __init__(self, log, name):
        object.__setattr__(self, '_log', log)
        object.__setattr__(self, '_name', name)
        object.__setattr__(self, '_kids', {})

    def __getattr__(self, k):
        if k.startswith('__') and k.endswith('__'):
            raise AttributeError(k)
        kids = object.__getattribute__(self, '_kids')
        if k not in kids:
            kids[k] = Rec(self._log, '%s.%s' % (self._name, k))
        return kids[k]

    def __setattr__(self, k, v):
        self._log.append(['set', '%s.%s' % (self._name, k), fmt(v)])

    def __setitem__(self, k, v):
        self._log.append(['setitem', self._name, fmt(k), fmt(v)])

    def __getitem__(self, k):
        return Rec(self._log, '%s[%s]' % (self._name, fmt(k)))

    def __call__(self, *a, **kw):
        self._log.append(['call', self._name, [fmt(x) for x in a], {k: fmt(v) for k, v in sorted(kw.items())}])
        return Rec(self._log, self._name + '()')

    def __enter__(self):
        return Rec(self._log, self._name + '.__enter__')

    def __exit__(self, *a):
        return False

    def __mul__(self, o):
        return Rec(self._log, '(%s*%s)' % (self._name, fmt(o)))

    __rmul__ = __mul__

    def __len__(self):
        return 3

    def __iter__(self):                                  # `row, col = A.getSizes()`
        return iter((self[0], self[1]))


def fmt(x):
    if isinstance(x, Rec):
        return '<%s>' % x._name
    if isinstance(x, (list, tuple)):
        return [fmt(v) for v in x]
    if isinstance(x, dict):
        return {str(k): fmt(v) for k, v in x.items()}
    if isinstance(x, np.ndarray):
        return ['ndarray'] + x.tolist()
    if callable(x):
        return 'callable:%s' % getattr(x, '__name__', type(x).__name__)
    if isinstance(x, (int, float, str, bool)) or x is None:
        return x
    return type(x).__name__


def load_reference_utils(log, root=REFERENCE):
    names = ['dolfinx', 'dolfinx.io', 'dolfinx.mesh', 'dolfinx.cpp', 'dolfinx.cpp.mesh', 'dolfinx.fem', 'dolfinx.fem.petsc',
             'dolfinx.nls', 'dolfinx.nls.petsc', 'dolfinx.la', 'ufl', 'petsc4py', 'mpi4py']
    stubs = {}
    for n in names:
        m = types.ModuleType(n)
        rec = Rec(log, n)
        m.__getattr__ = lambda k, rec=rec: getattr(rec, k)          # PEP 562: every name of the module is a recorder
        m.__path__ = []
        stubs[n] = m
    for n in names:                                                   # `from dolfinx import la` resolves submodules as attributes
        if '.' in n:
            parent, _, child = n.rpartition('.')
            setattr(stubs[parent], child, stubs[n])
    saved = {k: sys.modules.get(k) for k in stubs}
    sys.modules.update(stubs)
    try:
        spec = importlib.util.spec_from_file_location('_ref_utils_dolfinx', os.path.join(root, 'femo/fea/utils_dolfinx.py'))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mod


def record(root=REFERENCE):
    """name -> list of recorded events for each probed entry point of the reference's utils_dolfinx.py."""
    import contextlib
    import io
    log = []
    U = load_reference_utils(log, root)
    out = {}

    def probe(name, fn):
        del log[:]
        with contextlib.redirect_stdout(io.StringIO()):
            extra = fn()
        out[name] = [e for e in log]
        if extra is not None:
            out[name + ':result'] = extra
    F, w, bcs = Rec(log, 'F'), Rec(log, 'w'), Rec(log, 'bcs')
    probe('NewtonSolver(initialize=True)', lambda: U.NewtonSolver(F, w, bcs, initialize=True) and None)
    probe('NewtonSolver defaults', lambda: U.NewtonSolver(F, w, bcs) and None)

    def snes():
        U.SNESSolver(F, w, bcs)
        setf = [e for e in log if e[1].endswith('.setFunction')]
        return None
    probe('SNESSolver', snes)
    prob = U.NonlinearSNESProblem(F, w, bcs)
    x, b, Jm = Rec(log, 'x'), Rec(log, 'b'), Rec(log, 'J')
    probe('NonlinearSNESProblem.F', lambda: prob.F(None, x, b))
    probe('NonlinearSNESProblem.J', lambda: prob.J(None, x, Jm, None))
    probe('assembleSystem', lambda: U.assembleSystem(Rec(log, 'dRdu'), F, bcs=bcs) and None)
    probe('assembleMatrix', lambda: U.assembleMatrix(Rec(log, 'dRdu')) and None)
    probe('assembleVector', lambda: U.assembleVector(F) and None)
    probe('assemble bad dim', lambda: type(U.assemble(F, dim=3)).__name__)
    v = Rec(log, 'v')
    probe('update length 1', lambda: U.update(v, np.array([2.5])))
    probe('update array', lambda: U.update(v, np.array([1.0, 2.0, 3.0])))
    probe('solveNonlinear SNES', lambda: U.solveNonlinear(F, w, bcs, 'SNES', False, False))
    probe('solveNonlinear Newton', lambda: U.solveNonlinear(F, w, bcs, 'Newton', False, True))
    A = Rec(log, 'A')
    probe('solveKSP_mumps', lambda: U.solveKSP_mumps(A, b, x))
    probe('setUpKSP_MUMPS', lambda: U.setUpKSP_MUMPS(A) and None)
    probe('transpose', lambda: U.transpose(A) and None)
    probe('computeMatVecProductBwd', lambda: U.computeMatVecProductBwd(A, Rec(log, 'R')) and None)
    probe('createCustomMeasure ds', lambda: U.createCustomMeasure(Rec(log, 'mesh'), 1, Rec(log, 'marker'), 'ds', 100) and None)
    probe('project', lambda: U.project(Rec(log, 'expr'), Rec(log, 'target')))
    probe('project lumped', lambda: U.project(Rec(log, 'expr'), Rec(log, 'target'), lump_mass=True))
    out['DOLFIN_EPS'] = U.DOLFIN_EPS
    return out
