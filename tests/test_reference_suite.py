"""The reference's own test files, unmodified, against this package through ``blues_b200.compat`` (SURVEY.md §8(f)2).

The files come from the verbatim copies of MobleyLab/blues files under ``tests/golden/reference_checkout/`` (their
SHA-256 digests are pinned in ``tests/golden/reference_checkout_sha256.json``), or from a checkout named by
``BLUES_REFERENCE``.  The test file is copied to a temporary directory at run time because pytest would otherwise
import it as ``blues.tests.…`` from the checkout.  Without a GPU the host-side tests of
``blues/tests/test_simulation.py`` must pass as they are; every other test of that file must get as far as creating a
``Context`` and stop there with the engine's "no CUDA device … no CPU fallback" error — i.e. nothing is blocked by a
missing name or a different signature.
"""
import hashlib
import json
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHECKOUT = os.path.join(ROOT, 'tests', 'golden', 'reference_checkout')
REFERENCE = os.environ.get('BLUES_REFERENCE') or CHECKOUT

RUNNER = r'''
import sys
sys.dont_write_bytecode = True
sys.path.insert(0, %(root)r)
import blues_b200.compat as compat
compat.install(data_root=%(ref)r)
import pytest
sys.exit(pytest.main(['-p', 'no:cacheprovider', '-q', '-rA', '--tb=line', '--rootdir', %(tmp)r, '-c', '/dev/null', '--confcutdir', %(tmp)r, %(tmp)r]))
'''

HOST_ONLY = {
    'TestSystemFactory::test_atom_selections', 'TestSystemFactory::test_atomidx_to_atomlist',
    'TestSystemFactory::test_generateSystem', 'TestSystemFactory::test_generateAlchSystem',
    'TestSystemFactory::test_restrain_postions', 'TestSystemFactory::test_freeze_atoms',
    'TestSystemFactory::test_freeze_radius', 'TestSimulationFactory::test_addBarostat',
    'TestSimulationFactory::test_generateIntegrator', 'TestSimulationFactory::test_generateNCMCIntegrator',
}


def test_reference_test_simulation_runs_unmodified(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip('with a GPU the remaining tests of the file run too; this check is about the CPU container')
    shutil.copy(os.path.join(REFERENCE, 'blues', 'tests', 'test_simulation.py'), str(tmp_path))
    code = RUNNER % {'root': ROOT, 'ref': REFERENCE, 'tmp': str(tmp_path)}
    env = dict(os.environ, COLUMNS='400', PYTHONDONTWRITEBYTECODE='1')
    out = subprocess.run([sys.executable, '-c', code], cwd=str(tmp_path), env=env, capture_output=True, text=True,
                         timeout=600).stdout
    passed = set(re.findall(r'^PASSED \S*test_simulation\.py::(\S+)', out, re.M))
    blocked = re.findall(r'^(?:FAILED|ERROR) \S*test_simulation\.py::(\S+) - (.*)$', out, re.M)
    assert HOST_ONLY <= passed, (sorted(HOST_ONLY - passed), out[-3000:])
    assert len(passed) + len(blocked) == 25, out[-3000:]             # the file has 25 tests
    for name, why in blocked:
        assert 'no CUDA device available' in why and 'no CPU fallback' in why, (name, why)


ORACLE_RUNNER = r'''
import sys
sys.dont_write_bytecode = True
sys.path.insert(0, %(root)r)
import numpy
numpy.random.seed(1)                 # test_ethylene.py draws its integrator seeds from numpy's global generator
import blues_b200.compat as compat
compat.install(data_root=%(ref)r)
import blues_b200._native as native
from tests.oracle_engine import OracleEngine
native.Engine = OracleEngine            # test infrastructure: the C ABI's Python face answered by the CPU oracle
import pytest
sys.exit(pytest.main(['-p', 'no:cacheprovider', '-q', '-rA', '--tb=short', '--rootdir', %(tmp)r, '-c', '/dev/null', '--confcutdir', %(tmp)r, %(tmp)r]))
'''


def test_reference_tests_pass_on_the_host_layer_over_the_oracle_engine(tmp_path):
    """All 25 tests of ``test_simulation.py`` and ``test_randomrotation.py``, unmodified, against this package's host
    layer (SystemFactory … BLUESSimulation.run, YAML settings, reporters, the rotation move, state sync, accept/reject)
    with ``tests/oracle_engine.OracleEngine`` standing in for the CUDA engine below the C ABI.  Together with the
    ``-m gpu`` tests (CUDA engine == oracle on the same inputs) this is the reference's own acceptance test for the
    drop-in.  ``test_ethylene.py`` (the known-answer test: XML system of generic ``Custom*Force`` terms, NetCDF
    trajectories read back through the ``mdtraj`` alias, populations 0.25 / 0.75) runs the same way, the stand-in
    evaluating the ``custom_*`` tables with the host interpreter.  Not run: ``test_watertranslation.py`` (its
    ``eqToluene.prmtop`` is missing upstream), ``test_sidechain.py`` (OpenEye)."""
    for name in ('test_simulation.py', 'test_randomrotation.py', 'test_ethylene.py'):
        shutil.copy(os.path.join(REFERENCE, 'blues', 'tests', name), str(tmp_path))
    code = ORACLE_RUNNER % {'root': ROOT, 'ref': REFERENCE, 'tmp': str(tmp_path)}
    env = dict(os.environ, COLUMNS='400', PYTHONDONTWRITEBYTECODE='1')
    run = subprocess.run([sys.executable, '-c', code], cwd=str(tmp_path), env=env, capture_output=True, text=True,
                         timeout=1500)
    out = run.stdout
    passed = set(re.findall(r'^PASSED (\S+)', out, re.M))
    assert run.returncode == 0 and len(passed) == 28, out[-4000:]
    assert any('test_ethylene.py::test_runAnalysis' in p for p in passed)
    assert any('test_randomrotation.py' in p for p in passed)


def test_fixture_copies_are_verbatim():
    """tests/golden/reference_checkout/ (input of tests/test_gpu_reference_suite.py) is unchanged: each file matches the
    SHA-256 digest recorded for it in tests/golden/reference_checkout_sha256.json.  Where ``BLUES_REFERENCE`` names a
    checkout, its files must match the same digests, i.e. the copies equal that checkout byte for byte."""
    with open(os.path.join(ROOT, 'tests', 'golden', 'reference_checkout_sha256.json')) as fh:
        digests = json.load(fh)
    assert sorted(digests) == sorted(('test_simulation.py', 'test_randomrotation.py', 'test_ethylene.py',
                                      'data/TOL-parm.prmtop', 'data/TOL-parm.inpcrd', 'data/ethylene_system.xml',
                                      'data/ethylene_structure.pdb'))
    for base in sorted({CHECKOUT, REFERENCE}):
        for rel, want in digests.items():
            with open(os.path.join(base, 'blues', 'tests', rel), 'rb') as fh:
                assert hashlib.sha256(fh.read()).hexdigest() == want, (base, rel)
