"""CPU tests: host-side logic (units, parsers, system builder, bookkeeping pinned by the reference's own functions)."""
import json
import os
import re
import numpy as np
import pytest

from blues_b200 import unit as u
from blues_b200 import utils, lepton
from blues_b200.structure import Structure, AmberMask
from blues_b200.integrators import AlchemicalExternalLangevinIntegrator
from blues_b200.simulation import SystemFactory, SimulationFactory
from blues_b200.moves import uniform_quaternion, rotation_matrix_from_quaternion, select_atoms, MoveEngine, Move

GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')


@pytest.fixture(scope='module')
def tol():
    return Structure.load_npz(os.path.join(GOLDEN, 'tol_parm.npz'))


def test_unit_algebra():
    kT = u.MOLAR_GAS_CONSTANT_R * (300 * u.kelvin)
    assert abs(kT.value_in_unit(u.kilojoules_per_mole) - 2.494341741) < 1e-8
    assert (10 * u.angstroms).value_in_unit(u.nanometers) == pytest.approx(1.0)
    w = 5.0 * u.kilocalories_per_mole / u.angstroms ** 2
    assert w.value_in_unit(u.kilojoules_per_mole / u.nanometers ** 2) == pytest.approx(2092.0)
    p = u.Quantity(np.arange(12.0).reshape(4, 3), u.nanometers)
    assert p[[0, 2]].shape == (2, 3) and p[1].unit == u.nanometers
    p[0] = p[1]
    assert np.all(p._value[0] == p._value[1])
    assert utils.parse_unit_quantity('1 * 1/picoseconds').value_in_unit(u.picoseconds ** -1) == 1.0
    assert utils.parse_unit_quantity('3.024 * daltons').value_in_unit(u.dalton) == pytest.approx(3.024)
    e = 3 * u.kilojoules_per_mole
    assert isinstance(e * (-1.0 / kT), float)


def test_reference_bookkeeping_tables():
    """calculateNCMCSteps / _get_prop_lambda against outputs of the reference's own source (make_fixtures.py)."""
    tab = json.load(open(os.path.join(GOLDEN, 'reference_bookkeeping.json')))
    for (nsteps, nprop, pl), want in tab['calculateNCMCSteps']:
        assert utils.calculateNCMCSteps(nstepsNC=nsteps, nprop=nprop, propLambda=pl) == want
    integ = AlchemicalExternalLangevinIntegrator({'lambda_sterics': '1'})
    for pl, want in tab['get_prop_lambda']:
        assert list(integ._get_prop_lambda(pl)) == want


def test_ncmc_integrator_attributes():
    """blues/tests/test_simulation.py:262-289"""
    cfg = {'nstepsNC': 100, 'temperature': 100 * u.kelvin, 'dt': 0.001 * u.picoseconds, 'nprop': 2, 'propLambda': 0.1,
           'splitting': 'V H R O R H V', 'alchemical_functions': {'lambda_sterics': '1', 'lambda_electrostatics': '1'}}
    integ = SimulationFactory.generateNCMCIntegrator(**cfg)
    assert integ._n_steps_neq == 100
    assert integ._n_lambda_steps == 200
    assert integ._alchemical_functions == cfg['alchemical_functions']
    assert integ._splitting == 'V H R O R H V'
    assert integ._prop_lambda == (0.4, 0.6)
    assert integ.getTemperature().value_in_unit(u.kelvin) == 100
    assert integ.getStepSize().value_in_unit(u.picoseconds) == pytest.approx(0.001)
    assert integ.getGlobalVariableByName('nprop') == 2
    assert integ.getGlobalVariableByName('prop_lambda_min') == 0.4


def test_lambda_functions():
    fs = 'min(1, (1/0.3)*abs(lambda-0.5))'
    fe = 'step(0.2-lambda) - 1/0.2*lambda*step(0.2-lambda) + 1/0.2*(lambda-0.8)*step(lambda-0.8)'
    s, e = lepton.Expression(fs), lepton.Expression(fe)
    assert s(0.0) == 1 and s(0.5) == 0 and s(0.35) == pytest.approx(0.5) and s(1.0) == 1
    assert e(0.0) == 1 and e(0.1) == pytest.approx(0.5) and e(0.5) == 0 and e(0.9) == pytest.approx(0.5)
    assert lepton.tabulate('lambda^2', 4) == [0.0, 0.0625, 0.25, 0.5625, 1.0]
    with pytest.raises(ValueError):
        lepton.Expression('__import__("os")')


def test_prmtop_facts(tol):
    """SURVEY.md Appendix B: composition, term counts, charges, LJ known answers."""
    assert tol.n_atoms == 975 and len(tol.bonds) == 655 and len(tol.angles) == 344 and len(tol.dihedrals) == 36
    assert tol.residue_names[0] == 'LIG' and tol.residue_names.count('HOH') == 320
    assert np.sum(tol.charges ** 2) == pytest.approx(334.0509, abs=1e-3)
    assert abs(tol.charges.sum()) < 1e-6
    i = tol.atom_types.index('c3')
    assert tol.lj_sigma[i] * 0.1 == pytest.approx(0.339966951, rel=1e-7)
    assert tol.lj_epsilon[i] * 4.184 == pytest.approx(0.4577296, rel=1e-6)
    wd = Structure.load_npz(os.path.join(GOLDEN, 'wat_divaline.npz'))
    assert wd.n_atoms == 2591 and wd.velocities is not None
    ow = wd.atom_types.index('OW')
    assert wd.lj_sigma[ow] * 0.1 == pytest.approx(0.315075241, rel=1e-7)
    assert wd.lj_epsilon[wd.atom_types.index('HW')] == 0.0


def test_create_system(tol):
    system = tol.createSystem(nonbondedMethod='PME', nonbondedCutoff=8.0 * u.angstroms, constraints='HBonds')
    t = system.flatten()
    assert len(t['excl_pairs']) == 1026 and int((t['excl_eps'] != 0).sum()) == 27
    assert len(t['constraints']) == 8 + 3 * 320
    assert t['ewald_alpha'] == pytest.approx(3.28533, rel=1e-5) and list(t['pme_grid']) == [24, 24, 24]
    names = [type(f).__name__ for f in system.getForces()]
    assert names == ['HarmonicBondForce', 'HarmonicAngleForce', 'PeriodicTorsionForce', 'NonbondedForce', 'CMMotionRemover']
    s2 = tol.createSystem(nonbondedMethod='PME', nonbondedCutoff=10 * u.angstroms, ewaldErrorTolerance=0.005,
                          hydrogenMass=3.024 * u.dalton)
    assert s2.masses.sum() == pytest.approx(system.masses.sum())
    assert s2.flatten()['ewald_alpha'] == pytest.approx(2.14597, rel=1e-5)


def test_alchemical_system_and_factories(tol):
    """blues/tests/test_simulation.py:146-237 (structure of the systems; no GPU needed)."""
    idx = utils.atomIndexfromTop('LIG', tol.topology)
    assert idx == list(range(15))
    systems = SystemFactory(tol, idx, {'nonbondedMethod': 'PME', 'nonbondedCutoff': 8.0 * u.angstroms, 'constraints': 'HBonds'})
    md_forces = systems.md.getForces()
    alch_forces = systems.alch.getForces()
    assert len(alch_forces) > len(md_forces)
    assert any(type(f).__name__.startswith('Custom') for f in alch_forces)
    ta = systems.alch.flatten()
    assert np.all(ta['charge'][:15] == 0) and np.all(ta['epsilon'][:15] == 0) and len(ta['alch_exc_pairs']) == 27
    restrained = SystemFactory.restrain_positions(tol, systems.md, ':LIG')
    assert type(restrained.getForces()[-1]).__name__ == 'CustomExternalForce'
    flat = restrained.flatten()
    assert len(flat['restraint_atoms']) == 15
    assert np.all(flat['restraint_k'] == 5.0)          # 'k_restr' global parameter reaches the engine tables
    frozen = SystemFactory.freeze_atoms(tol, systems.alch, ':LIG')
    assert all(frozen.getParticleMass(i)._value == 0 for i in range(15))
    import copy
    fr = SystemFactory.freeze_radius(tol, copy.deepcopy(systems.md), freeze_distance=5 * u.angstrom,
                                     freeze_center=':LIG', freeze_solvent=':Cl-')
    sel = AmberMask(tol, '(:LIG<:5.0)&!(:Cl-)').Selection()
    assert [fr.getParticleMass(i)._value == 0 for i in range(975)] == [not bool(x) for x in sel]


def test_t4l_freeze_count():
    """docs/BLUES_tutorial.ipynb:718 — 22 065 atoms frozen by freeze_radius(':LIG', 5 A, ':HOH,Cl-')."""
    s = Structure.load_npz(os.path.join(GOLDEN, 't4l_surrogate.npz'))
    sel = AmberMask(s, '(:LIG<:5.000000)&!(:HOH,Cl-)').Selection()
    assert s.n_atoms - int(sel.sum()) == 22065


def test_move_helpers(tol):
    q = uniform_quaternion(3134)
    assert np.allclose(q, uniform_quaternion(3134)) and abs(np.dot(q, q) - 1) < 1e-12
    R = rotation_matrix_from_quaternion(q)
    assert np.allclose(R @ R.T, np.eye(3), atol=1e-12) and np.linalg.det(R) == pytest.approx(1.0)
    assert list(select_atoms(tol, '(index 3) or (index 5)')) == [3, 5]
    assert len(select_atoms(tol, 'resname LIG and not name C1')) == 14
    eng = MoveEngine([Move(), Move()], [1, 3])
    assert eng.probabilities == [0.25, 0.75]
    eng.selectMove()
    assert eng.move_name == 'Move'


def test_c_abi_library_exports_every_declared_symbol():
    """The shared library loads without a GPU and exports every function include/blues_b200.h declares."""
    import ctypes
    from blues_b200 import _native
    header = open(os.path.join(os.path.dirname(GOLDEN), '..', 'include', 'blues_b200.h')).read()
    declared = set(re.findall(r'\b(bl_[a-z_0-9]+)\s*\(', header))
    assert declared == set(_native.SYMBOLS), declared ^ set(_native.SYMBOLS)
    lib = _native.load_library()
    for name in declared:
        assert hasattr(lib, name)
    assert b'sm_100a' in lib.bl_version()
    assert ctypes.sizeof(_native.BlTopology) > 0


def test_ctypes_structs_match_the_c_header(tmp_path):
    """include/blues_b200.h is the contract: the ctypes mirrors in blues_b200/_native.py must have the same size and
    the same offset for every field (compiled with gcc from the header itself, no GPU needed)."""
    import ctypes
    import re
    import subprocess
    from blues_b200 import _native
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pairs = [('bl_topology', _native.BlTopology), ('bl_integrator_params', _native.BlIntegratorParams),
             ('bl_move', _native.BlMove)]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "blues_b200.h"', 'int main(void) {']
    for cname, cls in pairs:
        lines.append('printf("%s sizeof %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in cls._fields_:
            lines.append('printf("%s %s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines += ['return 0;', '}']
    src = tmp_path / 'layout.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'layout'
    subprocess.check_call(['gcc', '-std=c99', '-I', os.path.join(root, 'include'), str(src), '-o', str(exe)])
    out = subprocess.check_output([str(exe)], text=True)
    want = {}
    for line in out.splitlines():
        a, b, c = line.split()
        want[(a, b)] = int(c)
    for cname, cls in pairs:
        assert ctypes.sizeof(cls) == want[(cname, 'sizeof')], cname
        for fname, _ in cls._fields_:
            assert getattr(cls, fname).offset == want[(cname, fname)], (cname, fname)
    # every move kind the header defines is known to the binding
    hdr = open(os.path.join(root, 'include', 'blues_b200.h')).read()
    for name, value in re.findall(r'#define (BL_MOVE_\w+)\s+(\d+)', hdr):
        assert getattr(_native, name) == int(value), name


def test_restart_files_round_trip_ascii_and_netcdf(tmp_path):
    """RestartReporter (blues/reporters.py:224 asks parmed for NetCDF restarts) and the Rst7 reader behind the YAML
    `structure: restart:` key (blues/settings.py:76-85): both AMBER formats, detected by content."""
    from scipy.io import netcdf_file
    from blues_b200.reporters import RestartReporter, ReporterConfig
    from blues_b200.structure import Rst7, is_netcdf
    rs = np.random.RandomState(2)
    n = 37
    xyz = rs.uniform(0, 30, size=(n, 3))
    vel = rs.normal(size=(n, 3))
    box = np.diag([31.0, 32.5, 29.75])

    class FakeState(object):
        def getPositions(self, asNumpy=False):
            return u.Quantity(xyz.copy(), u.angstroms)

        def getVelocities(self, asNumpy=False):
            return u.Quantity(vel.copy(), u.angstroms / u.picoseconds)

        def getPeriodicBoxVectors(self, asNumpy=False):
            return u.Quantity(box.copy(), u.angstroms)

        def getTime(self):
            return u.Quantity(12.5, u.picoseconds)

    class FakeSystem(object):
        def getNumParticles(self):
            return n

    class FakeSim(object):
        system = FakeSystem()
        currentStep = 40

    for netcdf in (False, True):
        fname = str(tmp_path / ('r_%s.rst7' % netcdf))
        rep = RestartReporter(fname, reportInterval=10, netcdf=netcdf)
        assert rep.describeNextReport(FakeSim())[0] == 10 and rep.describeNextReport(FakeSim())[1:3] == (True, True)
        rep.report(FakeSim(), FakeState())
        assert is_netcdf(fname) == netcdf
        r = Rst7(fname)
        tol = 1e-12 if netcdf else 1e-6                       # the ASCII format keeps 7 decimals
        assert np.allclose(r.positions.value_in_unit(u.angstroms), xyz, atol=tol)
        assert np.allclose(r.velocities.value_in_unit(u.angstroms / u.picoseconds), vel, atol=30 * tol)
        assert np.allclose(r.box[:3], np.diag(box), atol=tol) and r.box[3:] == [90.0, 90.0, 90.0]
        assert r.hasvels and r.hasbox
    # AMBER NetCDF restart conventions (what parmed / cpptraj / sander expect to find)
    nc = netcdf_file(str(tmp_path / 'r_True.rst7'), 'r', mmap=False)
    assert nc.Conventions == b'AMBERRESTART' and nc.ConventionVersion == b'1.0'
    assert nc.variables['coordinates'].shape == (n, 3) and nc.variables['coordinates'].units == b'angstrom'
    assert nc.variables['velocities'].units == b'angstrom/picosecond'
    assert float(nc.variables['velocities'].scale_factor) == pytest.approx(20.455)
    assert np.allclose(nc.variables['velocities'][:] * 20.455, vel)
    assert nc.variables['time'].getValue() == pytest.approx(12.5)
    assert bytes(nc.variables['cell_angular'][:].tobytes()) == b'alphabeta gamma'
    assert np.allclose(nc.variables['cell_lengths'][:], np.diag(box))
    nc.close()
    # ReporterConfig follows the reference: restarts are NetCDF unless the YAML says otherwise
    reps = ReporterConfig(str(tmp_path / 'out'), {'restart': {'reportInterval': 5}}).makeReporters()
    assert isinstance(reps[0], RestartReporter) and reps[0].netcdf is True


def test_combination_move_orders_and_hooks():
    """blues/moves.py:1517-1560 (unrunnable upstream): members run in listed or reverse order, hooks fan out."""
    from blues_b200.moves import CombinationMove
    log = []

    class Rec(Move):
        def __init__(self, name, atoms):
            self.name, self.atom_indices = name, atoms

        def beforeMove(self, context):
            log.append(('before', self.name))
            return context

        def move(self, context):
            log.append(('move', self.name))
            return context + [self.name]

        def afterMove(self, context):
            log.append(('after', self.name))
            return context

    combo = CombinationMove([Rec('a', [1, 2]), Rec('b', [2, 3]), Rec('c', [7])])
    assert combo.atom_indices == [1, 2, 3, 7]
    np.random.seed(0)
    orders = set()
    for _ in range(40):
        out = combo.move([])
        assert out in (['a', 'b', 'c'], ['c', 'b', 'a'])
        orders.add(tuple(out))
    assert len(orders) == 2
    log.clear()
    assert combo.beforeMove('ctx') == 'ctx' and combo.afterMove('ctx') == 'ctx'
    assert log == [('before', 'a'), ('before', 'b'), ('before', 'c'), ('after', 'a'), ('after', 'b'), ('after', 'c')]
    eng = MoveEngine(combo)
    eng.selectMove()
    assert eng.move_name == 'CombinationMove' and eng.runEngine([]) in (['a', 'b', 'c'], ['c', 'b', 'a'])


class _FakeContext(object):
    """Positions in, positions out: what a host-path Move needs from a Context."""

    def __init__(self, xyz_nm):
        self.xyz = np.asarray(xyz_nm, float).copy()

    def getState(self, getPositions=False, **kw):
        ctx = self

        class S(object):
            def getPositions(self, asNumpy=False):
                return u.Quantity(ctx.xyz.copy(), u.nanometers)
        return S()

    def setPositions(self, pos):
        self.xyz = np.asarray(pos.value_in_unit(u.nanometers), float).copy()


def test_smart_dart_move(tol, tmp_path):
    """blues/moves.py:1086-1514: darts are ligand centres of mass stored in the frame of three basis particles; a
    ligand inside one dart jumps to another keeping its offset, follows the basis particles, and is left alone
    outside every dart; overlapping darts are an error."""
    from blues_b200.moves import SmartDartMove
    lig = [a.index for a in tol.topology.atoms() if a.residue.name == 'LIG']
    basis = [15, 18, 21]                                    # three water oxygens: not collinear
    shift = np.array([6.0, 0.0, 0.0])                       # Angstrom
    import copy
    other = copy.deepcopy(tol)
    c = np.array(tol.coordinates, float)
    c[lig] += shift
    other.coordinates = c
    # darts from Structure objects and from files give the same dartboard
    f1, f2 = str(tmp_path / 'a.pdb'), str(tmp_path / 'b.pdb')
    tol.save(f1, format='pdb')
    other.save(f2, format='pdb')
    mv = SmartDartMove(tol, basis, [tol, other], dart_radius=0.2 * u.nanometers)
    mv_files = SmartDartMove(tol, basis, [f1, f2], dart_radius=0.2 * u.nanometers)
    for a, b in zip(mv.n_dartboard, mv_files.n_dartboard):
        assert np.allclose(a.value_in_unit(u.nanometers), b.value_in_unit(u.nanometers), atol=2e-3)   # PDB: 3 decimals
    assert np.allclose(mv.dartboard[1].value_in_unit(u.nanometers) - mv.dartboard[0].value_in_unit(u.nanometers),
                       shift * 0.1, atol=1e-5)
    # frame algebra round trip
    p = np.array(tol.coordinates, float)[basis] * 0.1
    x = np.array([0.3, -0.2, 0.7])
    assert np.allclose(mv._findOldCoord(p[0], p[1], p[2], mv._findNewCoord(p[0], p[1], p[2], x)).value_in_unit(u.nanometers), x)
    # inside dart 0 (slightly off-centre): the ligand lands at dart 1 with the same offset, nothing else moves
    x0 = np.array(tol.coordinates, float) * 0.1
    off = np.array([0.05, -0.03, 0.02])
    x0[lig] += off
    ctx = _FakeContext(x0)
    assert mv.move(ctx) is ctx
    moved = ctx.xyz
    assert np.allclose(moved[lig] - x0[lig], shift * 0.1, atol=1e-5)
    rest = np.setdiff1d(np.arange(len(x0)), lig)
    assert np.array_equal(moved[rest], x0[rest])
    # and back again (two darts, self_dart False: the move is its own inverse)
    mv.move(ctx)
    assert np.allclose(ctx.xyz, x0, atol=1e-5)
    # the darts follow the basis particles: translate the whole system, the jump is unchanged
    ctx2 = _FakeContext(x0 + np.array([0.4, 0.1, -0.2]))
    mv.move(ctx2)
    assert np.allclose(ctx2.xyz[lig] - (x0[lig] + np.array([0.4, 0.1, -0.2])), shift * 0.1, atol=1e-5)
    # outside every dart: untouched
    far = x0.copy()
    far[lig] += np.array([0.0, 0.3, 0.0])
    ctx3 = _FakeContext(far)
    assert mv.move(ctx3) is ctx3 and np.array_equal(ctx3.xyz, far)
    # overlapping darts
    with pytest.raises(ValueError):
        mid = np.array(tol.coordinates, float) * 0.1
        mid[lig] += 0.5 * shift * 0.1                        # 0.3 nm from both dart centres
        SmartDartMove(tol, basis, [tol, other], dart_radius=0.4 * u.nanometers).move(_FakeContext(mid))
    with pytest.raises(ValueError):
        SmartDartMove(tol, basis, [tol])
    assert mv.device_move() is None


def test_committed_bench_line_keeps_the_contract():
    """profiles/r01_bench_1gpu.json is a line bench.py printed on a B200: every key of the bench contract is present
    and self-consistent (value = walkers x steps / time, roofline fraction = achieved / peak, e2e carries its bytes)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    line = json.load(open(os.path.join(root, 'profiles', 'r01_bench_1gpu.json')))
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'e2e', 'gpu_launches', 'clocks', 'roofline', 'cpu_baseline'):
        assert key in line, key
    assert line['n_gpus'] == 1 and line['warmup'] >= 3 and line['higher_is_better'] is True and line['scaling'] == 'weak'
    assert line['data'] == 'synthetic' and 'workload' in line['config'] and 'model' not in line['config']
    walkers = line['config']['global_walkers']
    assert line['value'] == pytest.approx(walkers * 1e3 / line['ms_per_step'], rel=1e-6)
    assert line['gpu_launches'] > line['steps']                      # several kernels per NCMC step
    e2e = line['e2e']
    assert e2e['unit'] == line['unit'] and e2e['h2d_bytes_per_step'] > 0 and e2e['d2h_bytes_per_step'] > 0
    assert 0 < e2e['value'] <= 1.02 * line['value']                  # host copies cannot make it faster
    roof = line['roofline']
    for key in ('bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'):
        assert key in roof, key
    assert roof['frac'] == pytest.approx(roof['achieved'] / roof['peak'], rel=1e-9) and 0 < roof['frac'] < 1
    cpu = line['cpu_baseline']
    assert cpu['kind'] in ('port', 'reference') and cpu['cores'] >= 1 and cpu['value'] > 0 and cpu['sample']
    assert not {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'} & set(line['clocks']['reasons'])
    assert line['clocks']['sm_mhz'] >= 0.9 * line['clocks']['sm_max_mhz']


def test_sidechain_rotor_perception_gives_the_chi_bonds_of_every_residue_type():
    """`SideChainMove` without OpenEye (blues/moves.py:418-843): backbone / ring / rotor perception from the bond graph
    must find exactly the side-chain torsion (chi) bonds of the standard residues — checked on one residue of each of the
    20 types of the T4 lysozyme surrogate topology (OpenEye's `IsRotor` on heavy-atom bonds gives the same set)."""
    from blues_b200.moves import SideChainMove
    s = Structure.load_npz(os.path.join(GOLDEN, 't4l_surrogate.npz'))
    chi = {'ALA': [], 'GLY': [], 'PRO': [], 'VAL': ['CA-CB'], 'SER': ['CA-CB'], 'THR': ['CA-CB'], 'CYS': ['CA-CB'],
           'LEU': ['CA-CB', 'CB-CG'], 'ILE': ['CA-CB', 'CB-CG1'], 'PHE': ['CA-CB', 'CB-CG'], 'TYR': ['CA-CB', 'CB-CG'],
           'TRP': ['CA-CB', 'CB-CG'], 'HIS': ['CA-CB', 'CB-CG'], 'ASP': ['CA-CB', 'CB-CG'], 'ASN': ['CA-CB', 'CB-CG'],
           'GLU': ['CA-CB', 'CB-CG', 'CG-CD'], 'GLN': ['CA-CB', 'CB-CG', 'CG-CD'], 'MET': ['CA-CB', 'CB-CG', 'CG-SD'],
           'LYS': ['CA-CB', 'CB-CG', 'CG-CD', 'CD-CE'], 'ARG': ['CA-CB', 'CB-CG', 'CG-CD', 'CD-NE']}
    names = [a.name for a in s.atoms]
    first = {}
    for r in list(s.topology.residues())[:164]:
        first.setdefault(r.name, int(r.id))
    assert set(first) == set(chi)
    for resname, rid in first.items():
        mv = SideChainMove(s, [rid])
        found = sorted('%s-%s' % (names[a], names[b]) for a, b in mv.rot_bonds)
        assert found == sorted(chi[resname]), (resname, rid, found)
        for bond, atoms in (mv.rot_atoms.get(rid) or {}).items():
            assert atoms[:2] == list(bond) and len(set(atoms)) == len(atoms)
            assert all(names[a] not in ('N', 'C', 'O') for a in atoms[2:])       # nothing of the backbone is rotated


def test_lepton_compiler_values_and_derivatives():
    """Custom*Force energy expressions -> stack programs (blues_b200/lepton.py): value and d/dr of the host twin of the
    device interpreter against direct evaluation and central differences, for every supported function."""
    import math
    from blues_b200 import lepton
    cases = [
        ('0.5*k*(r-r0)^2', {'k': 0, 'r0': 1}, {}, [250.0, 0.3], lambda r, p, g: 0.5 * p[0] * (r - p[1]) ** 2),
        ('4*eps*((s/r)^12-(s/r)^6); s=0.5*(s1+s2)*lambda_sterics; eps=sqrt(e1*e2)*lambda_electrostatics',
         {'s1': 0, 'e1': 1, 's2': 2, 'e2': 3}, {}, [0.3, 0.5, 0.34, 0.7],
         lambda r, p, g: 4 * math.sqrt(p[1] * p[3]) * g[1] * ((0.5 * (p[0] + p[2]) * g[0] / r) ** 12 - (0.5 * (p[0] + p[2]) * g[0] / r) ** 6)),
        ('A*exp(-b*r) - c/r^6 + step(r-0.4)*delta(0)*min(r, 0.5)*max(r, 0.1)', {'b': 0}, {'A': 1000.0, 'c': 0.002}, [12.0],
         lambda r, p, g: 1000.0 * math.exp(-p[0] * r) - 0.002 / r ** 6 + (1.0 if r >= 0.4 else 0.0) * min(r, 0.5) * max(r, 0.1)),
        ('q*erfc(a*r)/r + erf(r)*tanh(r) + sin(r)*cos(r)/tan(r+0.3) + log(r+1) + abs(r-0.5)^1.5 + select(r-0.2, sinh(r), cosh(r)) + atan(r)',
         {'q': 0}, {'a': 2.5}, [138.9],
         lambda r, p, g: p[0] * math.erfc(2.5 * r) / r + math.erf(r) * math.tanh(r) + math.sin(r) * math.cos(r) / math.tan(r + 0.3)
         + math.log(r + 1) + abs(r - 0.5) ** 1.5 + (math.sinh(r) if r - 0.2 != 0 else math.cosh(r)) + math.atan(r)),
        ('0.5*kc*distance(g1,g2)^2 + recip(distance(g1, g2)+1) + square(distance(g1,g2)) - cube(distance(g1,g2))', {'kc': 0}, {}, [1.0e5],
         lambda r, p, g: 0.5 * p[0] * r ** 2 + 1.0 / (r + 1) + r * r - r ** 3),
    ]
    for text, params, consts, par, ref in cases:
        ops, args = lepton.compile_program(text, params, consts, ['distance(g1,g2)'])
        for r in (0.27, 0.41, 0.66):
            for g in ((1.0, 1.0), (0.35, 0.8)):
                v, d = lepton.evaluate_program(ops, args, r, par, g)
                want = ref(r, par, g)
                fd = (ref(r + 1e-6, par, g) - ref(r - 1e-6, par, g)) / 2e-6
                assert abs(v - want) <= 1e-12 * max(1.0, abs(want)), (text, r, v, want)
                assert abs(d - fd) <= 2e-6 * max(1.0, abs(fd)), (text, r, d, fd)
    with pytest.raises(ValueError):
        lepton.compile_program('k*r + undefined_name', {'k': 0})
    with pytest.raises(ValueError):
        lepton.compile_program('a*r; a = b; b = a', {})
    with pytest.raises(NotImplementedError):
        lepton.compile_program('k*angle(g1,g2,g3)', {'k': 0})


def test_xml_system_round_trip_of_the_ethylene_known_answer_system():
    """XmlSerializer.deserialize on the reference's serialized System (verbatim fixture): particles, constraints, forces and
    the custom-force tables the engine receives."""
    from blues_b200.system import (XmlSerializer, CustomNonbondedForce, CustomCentroidBondForce, HarmonicBondForce,
                                   HarmonicAngleForce, PeriodicTorsionForce)
    xml = open(os.path.join(GOLDEN, 'reference_checkout', 'blues', 'tests', 'data', 'ethylene_system.xml')).read()
    system = XmlSerializer.deserialize(xml)
    assert system.getNumParticles() == 8 and system.getNumConstraints() == 4
    assert [system.getParticleMass(i)._value for i in range(3)] == [0.0, 0.0, 12.01]
    kinds = [type(f) for f in system.getForces()]
    assert kinds == [HarmonicBondForce, HarmonicAngleForce, PeriodicTorsionForce, CustomNonbondedForce, CustomCentroidBondForce]
    cn = system.getForces()[3]
    assert cn.getNumParticles() == 8 and cn.getNumInteractionGroups() == 1 and cn.getNumPerParticleParameters() == 4
    assert cn.global_params == {'lambda_sterics': 1.0, 'lambda_electrostatics': 1.0, 'lambda_charge': 1.0}
    cb = system.getForces()[4]
    assert cb.getNumGroups() == 2 and cb.getGroupParameters(0) == ([0, 1], [1.0, 1.0]) and cb.getGroupParameters(1) == ([2, 3], None)
    t = system.flatten()
    assert t['custom_term'].shape == (13, 4) and t['custom_n_params'] == 8 and len(t['custom_prog_start']) == 3
    assert list(t['custom_term'][-1][:2]) != list(t['custom_term'][0][:2])
    w = t['custom_group_weights']
    gs = t['custom_group_start']
    for k in range(len(gs) - 1):
        assert abs(w[gs[k]:gs[k + 1]].sum() - 1.0) < 1e-12                          # normalised group weights
    assert t['nb_method'] == 0 and np.allclose(t['box'], [2.0, 2.0, 2.0])


def test_trajectory_reader_distances_and_dihedrals(tmp_path):
    """blues_b200/trajectory.py (the ``mdtraj`` alias of compat): AMBER NetCDF in ångström → nm frames; distances with
    the minimum image; dihedral sign convention (IUPAC: trans = pi, right-handed twist positive)."""
    import math
    from scipy.io import netcdf_file
    from blues_b200 import trajectory
    x = np.array([[[0, 1, 0], [0, 0, 0], [1, 0, 0], [1, 0, 1]],
                  [[0, 1, 0], [0, 0, 0], [1, 0, 0], [1, -1, 0]],
                  [[0, 1, 0], [0, 0, 0], [19, 0, 0], [1, 1, 0]]], float)           # Å
    fn = str(tmp_path / 't.nc')
    nc = netcdf_file(fn, 'w', version=2)
    nc.createDimension('frame', None); nc.createDimension('spatial', 3); nc.createDimension('atom', 4)
    nc.createDimension('cell_spatial', 3); nc.createDimension('cell_angular', 3)
    nc.createVariable('time', 'f', ('frame',))
    nc.createVariable('coordinates', 'f', ('frame', 'atom', 'spatial'))
    nc.createVariable('cell_lengths', 'd', ('frame', 'cell_spatial'))
    nc.createVariable('cell_angles', 'd', ('frame', 'cell_angular'))
    for k in range(3):
        nc.variables['time'][k] = k
        nc.variables['coordinates'][k] = x[k]
        nc.variables['cell_lengths'][k] = [20.0, 20.0, 20.0]
        nc.variables['cell_angles'][k] = [90.0, 90.0, 90.0]
    nc.close()
    t = trajectory.load(fn)
    assert t.n_frames == 3 and t.n_atoms == 4 and len(t[1:]) == 2
    np.testing.assert_allclose(t.xyz, x * 0.1, atol=1e-6)
    d = trajectory.compute_distances(t, [[1, 2], [0, 3]])
    assert d.shape == (3, 2)
    np.testing.assert_allclose(d[:, 0], [0.1, 0.1, 0.1], atol=1e-6)                # frame 2: 1.9 nm wraps to 0.1 nm
    np.testing.assert_allclose(trajectory.compute_distances(t, [[1, 2]], periodic=False)[2, 0], 1.9, atol=1e-6)
    phi = trajectory.compute_dihedrals(t[:2], [[0, 1, 2, 3]])
    np.testing.assert_allclose(np.abs(phi[:, 0]), [math.pi / 2, math.pi], atol=1e-6)
    assert phi[0, 0] > 0            # seen along 1 -> 2 the front bond turns clockwise onto the back bond: +90 degrees


_STERICS = [1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 0.95, 0.8848447462380346, 0.8428373352131427, 0.7928373352131427,
            0.7490146003095886, 0.6934088361682191, 0.6515123083157823, 0.6088924298371354, 0.5588924298371354,
            0.5088924298371353, 0.4649556683144045, 0.4298606804827029, 0.3798606804827029, 0.35019373288005945,
            0.31648339779024653, 0.2780498882483276, 0.2521302239477468, 0.23139484523965026, 0.18729812232625365,
            0.15427643961733822, 0.12153116162972155, 0.09632462702545555, 0.06463743549588846, 0.01463743549588846, 0.0]
_STATICS = [1.0, 0.8519493439593149, 0.7142750443470669, 0.5385929179832776, 0.3891972949356391, 0.18820309596839535] + [0.0] * 26
# (schedule name, schedule, switching_types, steps) compared with golden/spread_lambda_protocol.json
SPREAD_LAMBDA_CASES = [(name, vals, kind, n) for name, vals, kind in (('sterics', _STERICS, 'sterics'),
                                                                      ('statics', _STATICS, 'auto'),
                                                                      ('statics', _STATICS, 'electrostatics'))
                       for n in (100, 37, 1000)]


def test_spread_lambda_protocol_and_tabulated_functions_in_the_integrator():
    """utils.spreadLambdaProtocol (blues/utils.py:276-369; the schedules are the ones of its docstring) and
    CustomIntegrator.addTabulatedFunction on the NCMC integrator: a symmetric protocol, plateaus exact, and the tables the
    engine receives are the tabulated functions sampled at every lambda step.  The values are compared with the tables
    stored in golden/spread_lambda_protocol.json and, where ``BLUES_REFERENCE`` names a checkout, with the reference's own
    function executed from its source text (its module cannot be imported here)."""
    import ast
    from blues_b200.lepton import Discrete1DFunction, Continuous1DFunction, Expression
    steps = 100
    st = utils.spreadLambdaProtocol(_STERICS, steps, switching_types='sterics', return_tab_function=False)
    el = utils.spreadLambdaProtocol(_STATICS, steps, switching_types='auto', return_tab_function=False)
    for tab in (st, el):
        assert len(tab) == steps + 1 and tab[0] == 1.0 and tab[-1] == 1.0 and abs(tab[steps // 2]) < 1e-12
        assert all(0.0 <= v <= 1.0 for v in tab)
        np.testing.assert_allclose(tab, tab[::-1], atol=1e-12)                     # symmetric about the midpoint
    assert st[:10] == [1.0] * 10 and el[12:50] == [0.0] * 38                       # plateaus restored exactly
    assert el[1] < 1.0 and st[9] == 1.0 and st[10] < 1.0                           # electrostatics go first
    with pytest.raises(ValueError):
        utils.spreadLambdaProtocol(_STATICS, steps, switching_types='bogus')
    with open(os.path.join(GOLDEN, 'spread_lambda_protocol.json')) as fh:
        golden = json.load(fh)['tables']
    assert sorted(golden) == sorted('%s/%s/%d' % (name, kind, n) for name, _, kind, n in SPREAD_LAMBDA_CASES)
    for name, vals, kind, n in SPREAD_LAMBDA_CASES:
        got = utils.spreadLambdaProtocol(list(vals), n, switching_types=kind, return_tab_function=False)
        np.testing.assert_allclose(got, golden['%s/%s/%d' % (name, kind, n)], rtol=0, atol=1e-12)
    ref_src = os.path.join(os.environ.get('BLUES_REFERENCE') or os.devnull, 'blues', 'utils.py')
    if os.path.exists(ref_src):
        tree = ast.parse(open(ref_src).read())
        fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == 'spreadLambdaProtocol'][0]
        from math import floor
        from scipy.interpolate import interp1d
        ns = {'np': np, 'interp1d': interp1d, 'floor': floor}
        exec(compile(ast.Module([fn], []), ref_src, 'exec'), ns)
        for _, vals, kind, n in SPREAD_LAMBDA_CASES:
            want = ns['spreadLambdaProtocol'](list(vals), n, switching_types=kind, return_tab_function=False)
            got = utils.spreadLambdaProtocol(list(vals), n, switching_types=kind, return_tab_function=False)
            np.testing.assert_allclose(got, want, rtol=0, atol=1e-12)
    # tabulated functions
    f = utils.spreadLambdaProtocol(_STERICS, steps, switching_types='sterics')
    assert isinstance(f, Discrete1DFunction) and f(0) == 1.0 and f(50.4) == f(50) and f(-1) == 0.0 and f(101) == 0.0
    c = Continuous1DFunction([0.0, 1.0, 4.0, 9.0], 0.0, 3.0)
    assert abs(c(2.0) - 4.0) < 1e-12 and c(3.5) == 0.0 and 1.0 < c(1.5) < 4.0
    assert Expression('2*tab(lambda*100)', {'tab': f})(0.5) == 2 * f(50)
    with pytest.raises(ValueError):
        Expression('tab(lambda)')                                                  # unknown function without the table
    integ = AlchemicalExternalLangevinIntegrator(
        alchemical_functions={'lambda_sterics': 'sterics_tab(lambda*100)', 'lambda_electrostatics': 'elec_tab(lambda*100)'},
        splitting='H V R O R V H', nsteps_neq=50)
    assert integ.addTabulatedFunction('sterics_tab', f) == 0
    assert integ.addTabulatedFunction('elec_tab', Discrete1DFunction(el)) == 1
    assert integ.getNumTabulatedFunctions() == 2 and integ.getTabulatedFunctionName(1) == 'elec_tab'
    ls, le = integ._tables()                                                       # 2 H steps x 50 = 100 lambda steps
    np.testing.assert_allclose(ls, st, atol=0)
    np.testing.assert_allclose(le, el, atol=0)
