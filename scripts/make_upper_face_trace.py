"""Runs the reference's own upper layer (femo/fea/fea_dolfinx.py FEA, femo/csdl_opt/*.py operations and FEAModel, imported
unmodified from the checkout $FEMO_REFERENCE names) over the recording stub lower face of tests/_upper_face.py and stores every lower-face call and
every value the callbacks write as tests/golden/upper_face_trace.json.  tests/test_upper_face.py holds femo_b200's mirrors to it.

    FEMO_REFERENCE=<reference checkout> python scripts/make_upper_face_trace.py
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import _upper_face as U   # noqa: E402

if not U.REFERENCE:
    sys.exit('set FEMO_REFERENCE to a checkout of the reference femo project')

world = U.World()
trace = U.scenario(world, U.load_reference(world))
path = os.path.join(ROOT, 'tests', 'golden', 'upper_face_trace.json')
with open(path, 'w') as f:
    json.dump(trace, f, indent=0)
print('%d steps -> %s' % (len(trace), path))
