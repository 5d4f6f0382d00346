"""Upper face of the drop-in boundary (SURVEY.md section 8b) held to the REFERENCE'S OWN CODE: tests/golden/upper_face_trace.json
is a run of femo's unmodified `FEA`, `StateOperation`, `OutputOperation`, `OutputFieldOperation` and `FEAModel`
(/root/reference/femo/fea/fea_dolfinx.py:70-234, femo/csdl_opt/*.py) over the recording stub lower face of tests/_upper_face.py
(scripts/make_upper_face_trace.py).  femo_b200's mirrors, run over the same stub, must make the same lower-face calls in the
same order with the same arrays and write the same values into the CSDL containers -- except for the documented quirks
they diverge from on purpose (DESIGN.md section 4): B8 (one assembly pass for dR/du and the BC'd system matrix), B4 (the
reference's forward solve passes the transposed operator with swapped vectors and returns zeros) and B3 (the reference
reuses the KSP of A for the adjoint).  No GPU, no engine, no oracle involved."""
import json
import os

import pytest

import _upper_face as U

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'upper_face_trace.json')
DRDU = ['assembleMatrix', 'd(R(u,f))/d(u0)', 0]


@pytest.fixture(scope='module')
def reference():
    with open(GOLD) as f:
        return {s[0]: s for s in json.load(f)}


@pytest.fixture(scope='module')
def mirror():
    world = U.World()
    with U.patched(world) as impl:
        run = U.scenario(world, impl)
    return {s[0]: json.loads(json.dumps(s)) for s in run}


def test_fixture_is_what_the_reference_does_today(reference):
    """Where $FEMO_REFERENCE names a reference checkout the committed trace is regenerated from it."""
    if not U.REFERENCE or not os.path.isdir(os.path.join(U.REFERENCE, 'femo')):
        pytest.skip('no reference checkout')
    world = U.World()
    live = json.loads(json.dumps(U.scenario(world, U.load_reference(world))))
    assert [s[0] for s in live] == list(reference)
    for s in live:
        assert s == reference[s[0]], s[0]


IDENTICAL = ['registry', 'registry-keys', 'StateOperation.define', 'evaluate_residuals', 'solve_residual_equations',
             'custom_solve twice', 'compute_jacvec_product fwd', 'compute_jacvec_product fwd, absent keys',
             'compute_jacvec_product rev', 'compute_jacvec_product rev, absent keys', 'apply_inverse_jacobian rev linear=False',
             'OutputOperation.compute', 'OutputOperation.compute_derivatives', 'OutputFieldOperation.compute', 'FEAModel run']


@pytest.mark.parametrize('name', IDENTICAL)
def test_identical_calls_and_values(reference, mirror, name):
    """Registry contents (keys, shapes, partial forms, attributes, the duplicate-input error, quirk B5's overwrite), every
    callback's lower-face calls and every value written: equal to the reference's, event for event and bit for bit."""
    assert mirror[name][1] == reference[name][1]
    assert mirror[name][2] == reference[name][2]


def test_step_list_is_complete(reference, mirror):
    assert list(mirror) == list(reference)
    assert set(reference) == set(IDENTICAL) | {'compute_derivatives', 'FEAModel compute_totals', 'apply_inverse_jacobian fwd linear=False',
                                              'apply_inverse_jacobian fwd linear=True', 'apply_inverse_jacobian rev linear=True'}


@pytest.mark.parametrize('name', ['compute_derivatives', 'FEAModel compute_totals'])
def test_linearisation_differs_only_by_the_merged_assembly(reference, mirror, name):
    """Quirk B8: the reference assembles dR/du twice (assembleMatrix, then assembleSystem with the BCs, state_model.py:132,149);
    the mirror takes both from one assembleSystem pass.  Same calls otherwise, same values handed to CSDL."""
    ref, mir = reference[name][1], mirror[name][1]
    assert ref.count(DRDU) == 1 and mir.count(DRDU) == 0
    assert sorted(map(json.dumps, [e for e in ref if e != DRDU])) == sorted(map(json.dumps, mir))
    assert sum(e[0] == 'assembleSystem' for e in mir) == 1
    assert mirror[name][2] == reference[name][2]


@pytest.mark.parametrize('linear', [False, True])
def test_forward_solve_is_the_intended_one(reference, mirror, linear):
    """Quirk B4 (fea_dolfinx.py:192-206), seen by running the reference: it solves INTO dR with du = 0 as the right-hand side
    and returns du, i.e. zeros.  The mirror solves A du = dR."""
    name = 'apply_inverse_jacobian fwd linear=%s' % linear
    ref, mir = reference[name], mirror[name]
    assert all(v == 0.0 for v in ref[2]['d_outputs']['u'])
    assert any(v != 0.0 for v in mir[2]['d_outputs']['u'])
    assert mir[2]['d_residuals'] == ref[2]['d_residuals']                 # the seed is left alone by both
    assert [e[0] for e in mir[1]] == [e[0] for e in ref[1]]               # same steps: set dR, zero du, one solve, read du
    solve_ref, solve_mir = ref[1][2], mir[1][2]
    dR, du = ref[1][0][1], ref[1][1][1]
    assert solve_ref[2:] == [du, '0.0/4', dR]                             # reference: b = du (zeros), x = dR
    assert solve_mir[2] == dR and solve_mir[4] == du                      # mirror: b = dR, x = du
    assert solve_mir[1] == 'A[d(R(u,f))/d(u0)|2]'                         # ... with A itself, not its transpose


def test_adjoint_solve_with_a_kept_factorisation_uses_the_transpose(reference, mirror):
    """Quirk B3 (fea_dolfinx.py:208-222 with linear_problem): the reference applies the KSP of A to the adjoint right-hand
    side (valid for symmetric A only); the mirror always solves with the true transpose.  Same vectors in, same slot out."""
    name = 'apply_inverse_jacobian rev linear=True'
    ref, mir = reference[name][1], mirror[name][1]
    assert [e for e in ref if e[0] not in ('ksp.solve',)] == [e for e in mir if e[0] not in ('solveKSP_mumps',)]
    (kr,), (km,) = [e for e in ref if e[0] == 'ksp.solve'], [e for e in mir if e[0] == 'solveKSP_mumps']
    assert kr[1] == 'A[d(R(u,f))/d(u0)|2]' and km[1] == 'T(A[d(R(u,f))/d(u0)|2])'
    assert kr[2:] == km[2:]


def test_output_partials_survive_the_staging_ring():
    """The lower face hands vectors out of a ring of three staging buffers per size; an output with more than three same-size
    arguments must still deliver intact partials to a backend that keeps references (advisor finding, round 1)."""
    import numpy as np
    from femo_b200.csdl_opt import output_model as om
    ring = [np.zeros(5) for _ in range(3)]
    calls = []

    def assemble(form, dim=0):
        buf = ring[len(calls) % 3]
        buf[:] = len(calls) + 1.0
        calls.append(form)
        return buf
    world = U.World()
    saved = {k: om.__dict__[k] for k in ('assemble', 'computePartials', 'update')}
    om.assemble, om.computePartials, om.update = assemble, (lambda form, f: (form, f.name)), (lambda f, a: None)
    try:
        fea = type('F', (), {})()
        args = {n: dict(function=world.Function(world.Space(5), n), shape=5) for n in 'abcde'}
        fea.outputs_dict = {'J': dict(form='J', shape=1)}
        op = om.OutputOperation(fea=fea, args_dict=args, output_name='J')
        d = {}
        op.compute_derivatives({n: np.zeros(5) for n in args}, d)
    finally:
        om.__dict__.update(saved)
    assert [float(d['J', n][0]) for n in 'abcde'] == [1.0, 2.0, 3.0, 4.0, 5.0]
    calls.clear()
    om.assemble, om.computePartials, om.update = assemble, (lambda form, f: (form, f.name)), (lambda f, a: None)
    try:
        op = om.OutputOperation(fea=fea, args_dict={n: args[n] for n in 'ab'}, output_name='J')
        d = {}
        op.compute_derivatives({n: np.zeros(5) for n in 'ab'}, d)
    finally:
        om.__dict__.update(saved)
    assert d['J', 'a'] is ring[0] and d['J', 'b'] is ring[1]            # up to three partials stay copy-free
