"""femo_b200.compat: the reference's import lines resolve to the B200 engine (no GPU)."""
import subprocess
import sys
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(code):
    out = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    return out.stdout


def test_reference_import_lines_resolve_to_the_mirrors():
    """The import lines of the reference's examples/*/run_*.py (`from femo.fea.fea_dolfinx import *`,
    `from femo.csdl_opt.fea_model import FEAModel`, ...) after `femo_b200.compat.install()`; run in a fresh interpreter
    so that the aliases do not leak into the other tests."""
    out = _run('''
import femo_b200.compat as c
names = c.install()
assert 'femo.fea.fea_dolfinx' in names and 'femo.csdl_opt.fea_model' in names
from femo.fea.fea_dolfinx import *
from femo.csdl_opt.fea_model import FEAModel
from femo.csdl_opt.state_model import StateModel, StateOperation
from femo.csdl_opt.output_model import OutputModel, OutputFieldModel
import femo.fea.utils_dolfinx as u
import femo_b200.fea.fea_b200 as fb, femo_b200.csdl_opt.fea_model as fm
assert FEA is fb.FEA and FEAModel is fm.FEAModel and u.update is update
mesh = createUnitSquareMesh(4)
fea = FEA(mesh)
f = Function(FunctionSpace(mesh, ('DG', 0)))
fea.add_input('f', f)
assert fea.inputs_dict['f']['shape'] == 32 and getFuncArray(f).min() == 1.0
c.uninstall()
import sys
assert not any(k == 'femo' or k.startswith('femo.') for k in sys.modules)
print('ok')
''')
    assert out.strip().endswith('ok')


def test_lower_face_only():
    """install(csdl_opt=False): only the modules femo's own csdl_opt package imports are aliased."""
    out = _run('''
import sys, femo_b200.compat as c
names = c.install(csdl_opt=False)
assert 'femo.fea.fea_dolfinx' in names and not any(n.startswith('femo.csdl_opt') for n in names)
assert 'femo.csdl_opt' not in sys.modules
print('ok')
''')
    assert out.strip().endswith('ok')


def test_reference_csdl_layer_defines_over_the_real_lower_face():
    """femo's OWN femo/csdl_opt package (loaded unmodified from the reference checkout, csdl replaced by the stand-in base
    classes) on top of femo_b200.fea through the aliases: FEAModel -> StateModel / OutputModel -> operations are defined for
    the nonlinear Poisson example's registry, with the shapes the engine's spaces report.  (Running the callbacks needs the
    GPU; their call sequence against the lower face is pinned in tests/test_upper_face.py.)"""
    ref = os.path.abspath(os.environ['FEMO_REFERENCE']) if os.environ.get('FEMO_REFERENCE') else ''
    if not ref or not os.path.isdir(os.path.join(ref, 'femo')):
        import pytest
        pytest.skip('no reference checkout')
    out = _run('''
REF = %r
import os, sys, types, importlib.util
import femo_b200.compat as c
c.install(csdl_opt=False)
from femo_b200.csdl_opt import _csdl_compat as cc
csdl = types.ModuleType('csdl')
csdl.Model, csdl.CustomImplicitOperation, csdl.CustomExplicitOperation, csdl.custom = cc.Model, cc.CustomImplicitOperation, cc.CustomExplicitOperation, cc.csdl.custom
sys.modules['csdl'] = csdl
pkg = types.ModuleType('femo.csdl_opt'); pkg.__path__ = [os.path.join(REF, 'femo', 'csdl_opt')]; sys.modules['femo.csdl_opt'] = pkg
from femo.csdl_opt.fea_model import FEAModel                 # the reference's file
import femo.csdl_opt.state_model as sm
assert sm.__file__.startswith(os.path.join(REF, ''))
from femo.fea.fea_dolfinx import *
from femo_b200.forms.nonlinear_poisson import pdeRes, outputForm
mesh = createUnitSquareMesh(6)
fea = FEA(mesh)
f = Function(FunctionSpace(mesh, ('DG', 0))); u = Function(FunctionSpace(mesh, ('CG', 1)))
fea.add_input('f', f)
fea.add_state(name='u', function=u, residual_form=pdeRes(u, TestFunction(u.function_space), f), arguments=['f'])
fea.add_output(name='l2_functional', type='scalar', form=outputForm(u, f), arguments=['f', 'u'])
model = FEAModel(fea=[fea])
sim = cc.Simulator(model, pinned=False)
ops = [(type(op).__module__, type(op).__name__, args, out) for op, args, out in model.ops]
assert ops == [('femo.csdl_opt.state_model', 'StateOperation', ['f'], 'u'),
               ('femo.csdl_opt.output_model', 'OutputOperation', ['f', 'u'], 'l2_functional')], ops
assert sim.vars['f'].shape == (72,) and sim.vars['u'].shape == (49,) and sim.vars['l2_functional'].shape == (1,)
print('ok')
''' % ref)
    assert out.strip().endswith('ok')
