"""Records what the reference's own femo/fea/utils_dolfinx.py (imported unmodified from the checkout $FEMO_REFERENCE names) asks dolfinx / PETSc
to do -- solver types, tolerances, lifting conventions, ... -- over the recording stand-in of tests/_lower_face.py, as
tests/golden/lower_face_calls.json.  tests/test_lower_face.py holds the oracle and the engine's defaults to it.

    FEMO_REFERENCE=<reference checkout> python scripts/make_lower_face_calls.py
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import _lower_face as L   # noqa: E402

if not L.REFERENCE:
    sys.exit('set FEMO_REFERENCE to a checkout of the reference femo project')

path = os.path.join(ROOT, 'tests', 'golden', 'lower_face_calls.json')
rec = L.record()
with open(path, 'w') as f:
    json.dump(rec, f, indent=0)
print('%d probes -> %s' % (len(rec), path))
