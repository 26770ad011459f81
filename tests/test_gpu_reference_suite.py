"""The reference's own test files, unmodified, against the CUDA engine (SURVEY.md §8(f)2; VERDICT r1 item 8).

``blues/tests/test_simulation.py`` (25 tests: SystemFactory, SimulationFactory, BLUESSimulation incl. ``run``, state sync,
accept/reject, YAML), ``blues/tests/test_randomrotation.py`` and ``blues/tests/test_ethylene.py`` (the reference's
known-answer test of the NCMC protocol: two-state populations 0.25 / 0.75) are kept verbatim as fixtures under
``tests/golden/reference_checkout/`` together with the TOL-parm files they read (the checkout itself does not exist on
the GPU box).  They are copied to a temporary directory, ``blues_b200.compat`` provides the ``blues`` / ``simtk`` /
``parmed`` / ``mdtraj`` names they import, and pytest runs them in a subprocess: every ``Context`` they create is a CUDA engine handle
behind the C ABI — no oracle, no stand-in.
"""
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHECKOUT = os.path.join(ROOT, 'tests', 'golden', 'reference_checkout')

RUNNER = r'''
import sys
sys.dont_write_bytecode = True
sys.path.insert(0, %(root)r)
import numpy
numpy.random.seed(%(seed)d)          # test_ethylene.py draws its integrator seeds from numpy's global generator
import blues_b200.compat as compat
compat.install(data_root=%(ref)r)
import blues_b200._native as native
assert native.Engine.__module__ == 'blues_b200._native'      # the real engine class, not a stand-in
import pytest
rc = pytest.main(['-p', 'no:cacheprovider', '-q', '-rA', '--tb=short', '--rootdir', %(tmp)r, '-c', '/dev/null', '--confcutdir', %(tmp)r, %(tmp)r])
print('ENGINES_CREATED', native.Engine.created if hasattr(native.Engine, 'created') else -1)
sys.exit(rc)
'''


@pytest.mark.gpu
def test_reference_test_files_pass_unmodified_on_the_cuda_engine(tmp_path):
    for name in ('test_simulation.py', 'test_randomrotation.py'):
        shutil.copy(os.path.join(CHECKOUT, 'blues', 'tests', name), str(tmp_path))
    code = RUNNER % {'root': ROOT, 'ref': CHECKOUT, 'tmp': str(tmp_path), 'seed': 1}
    env = dict(os.environ, COLUMNS='400', PYTHONDONTWRITEBYTECODE='1', OMM_PLATFORM='CUDA')
    run = subprocess.run([sys.executable, '-c', code], cwd=str(tmp_path), env=env, capture_output=True, text=True,
                         timeout=1500)
    out = run.stdout
    passed = set(re.findall(r'^PASSED (\S+)', out, re.M))
    failed = re.findall(r'^(?:FAILED|ERROR) (\S+)', out, re.M)
    assert run.returncode == 0 and not failed and len(passed) == 26, (failed, out[-4000:], run.stderr[-2000:])
    assert any('test_randomrotation.py' in p for p in passed)
    m = re.search(r'ENGINES_CREATED (-?\d+)', out)
    assert m and int(m.group(1)) > 0, 'the reference tests must have created CUDA engine handles'


@pytest.mark.gpu
def test_reference_ethylene_known_answer_test_passes_unmodified_on_the_cuda_engine(tmp_path):
    """``blues/tests/test_ethylene.py`` as it is: 5 runs x 100 iterations of 20 NCMC + 20 MD steps on the XML system of
    generic Custom*Force terms, NetCDF trajectories through ``ReporterConfig``, read back with ``mdtraj.load`` /
    ``compute_distances``; populations of the two states must come out 0.25 / 0.75 within the test's own error bar.
    numpy's generator is seeded by the runner, so the whole run is reproducible (the engine is bitwise deterministic)."""
    shutil.copy(os.path.join(CHECKOUT, 'blues', 'tests', 'test_ethylene.py'), str(tmp_path))
    code = RUNNER % {'root': ROOT, 'ref': CHECKOUT, 'tmp': str(tmp_path), 'seed': 1}
    env = dict(os.environ, COLUMNS='400', PYTHONDONTWRITEBYTECODE='1', OMM_PLATFORM='CUDA')
    run = subprocess.run([sys.executable, '-c', code], cwd=str(tmp_path), env=env, capture_output=True, text=True,
                         timeout=1500)
    out = run.stdout
    passed = set(re.findall(r'^PASSED (\S+)', out, re.M))
    failed = re.findall(r'^(?:FAILED|ERROR) (\S+)', out, re.M)
    assert run.returncode == 0 and not failed and len(passed) == 2, (failed, out[-4000:], run.stderr[-2000:])
    m = re.search(r'ENGINES_CREATED (-?\d+)', out)
    assert m and int(m.group(1)) >= 15, 'md, alch and ncmc contexts of 5 runs must be CUDA engine handles'
    for k in range(5):
        assert os.path.getsize(os.path.join(str(tmp_path), 'ethylene-test_%d.nc' % k)) > 0
