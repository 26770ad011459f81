#!/usr/bin/env python
"""Run the reference's own test files, unmodified, against blues_b200 through the import shim.

    python tools/run_reference_tests.py /path/to/MobleyLab/blues [--oracle-engine] [pytest args …]

Copies ``blues/tests/test_simulation.py`` and ``test_randomrotation.py`` of the checkout to a temporary directory
(pytest would otherwise import them as ``blues.tests.*`` from the checkout itself), installs ``blues_b200.compat``
with the checkout as data root, and runs pytest there.  On a machine with a B200 the whole of both files runs; without
a GPU only the host-side tests do (``tests/test_reference_suite.py`` asserts exactly that split) — unless
``--oracle-engine`` puts the CPU oracle behind the engine interface (test infrastructure, ``tests/oracle_engine.py``),
with which all 26 tests pass on a CPU.  Not included:
``test_watertranslation.py`` (its ``eqToluene.prmtop`` is missing upstream), ``test_ethylene.py`` (generic
``Custom*Force`` expressions from a serialized OpenMM system), ``test_sidechain.py`` (OpenEye toolkits).
"""
import os
import shutil
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main(argv):
    if len(argv) < 2:
        print(__doc__)
        return 2
    ref = os.path.abspath(argv[1])
    sys.dont_write_bytecode = True
    sys.path.insert(0, ROOT)
    os.environ.setdefault('OMM_PLATFORM', 'CUDA')
    import blues_b200.compat as compat
    compat.install(data_root=ref)
    args = argv[2:]
    if '--oracle-engine' in args:
        args.remove('--oracle-engine')
        import blues_b200._native as native
        from tests.oracle_engine import OracleEngine
        native.Engine = OracleEngine
    import pytest
    tmp = tempfile.mkdtemp(prefix='blues_ref_tests_')
    for name in ('test_simulation.py', 'test_randomrotation.py'):
        shutil.copy(os.path.join(ref, 'blues', 'tests', name), tmp)
    os.chdir(tmp)
    return pytest.main(['-p', 'no:cacheprovider', '--rootdir', tmp, '-c', '/dev/null', '--confcutdir', tmp, tmp] + args)


if __name__ == '__main__':
    sys.exit(main(sys.argv))
