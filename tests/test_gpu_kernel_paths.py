"""The engine's force kernels against the float64 oracle on the paths the parity tests do not reach.

A host query (get_forces / get_energy / get_energy_terms) runs an *energy* evaluation.  Most forces of a run come from
*force-only* evaluations: every MD step and every evaluation inside an NCMC step except the last of a call.  For PME
those run the packed-FP32 pair kernel k_pair4 with its own Ewald fit (degree 10 up to zmax = 1.02 (alpha r_c)^2 = 4.8,
12 up to 11.5, the erfc form beyond) and the force-only reciprocal-space kernels.  More than two walkers switch the PME
spread / gather kernels and the list builder's configuration.

After md_run the engine holds the force-only forces at exactly the positions they were evaluated at (no frozen atoms:
no partial rows), so get_positions / get_forces read them; a following get_energy re-evaluates on the energy path at
the same positions.  Every walker is compared with the oracle at its own coordinates, with the limits of
test_gpu_parity.py.  At such unrounded coordinates a few pairs sit within float32 rounding of the cutoff; their atoms
are left out of the force comparison (cutoff_edge_atoms).  Every sum on the device is fixed point, so which slot a
walker occupies must not change a bit.
"""
import numpy as np
import pytest

from blues_b200 import unit as u
from tests.gpu_checks import ORACLE_TERMS, lambda_tables, load_case, rel_force_error

FORCE_TOL = 1e-4      # max over atoms of |dF| / max(|F_atom|, rms|F|)   (test_gpu_parity.py)
ENERGY_TOL = 1e-4     # relative, on the total potential energy
C_ORACLE_ABOVE = 5000  # atoms: above this the oracle's C twin (same formulas, OpenMP) replaces the numpy oracle
ZMAX_DEG10, ZMAX_FIT_TOP = 4.8, 11.5   # Ewald-fit regimes of k_pair4 (engine.cu, bl_create)
EDGE = 1e-6           # nm: float32 rounding of a distance near the cutoff (cutoff_edge_atoms)
ALCH_TERMS = ('alch_sterics', 'alch_electrostatics', 'alch_exceptions')
RF = dict(nonbondedMethod='CutoffPeriodic', nonbondedCutoff=9.0 * u.angstroms)
# fixtures whose coordinates clash (tol_parm: ~1.7e7 kJ/mol of direct-space energy): one MD step from them throws atoms
# nanometres, so their walkers start from a relaxed frame (as the parity tests' trajectories of tol_parm do)
MINIMIZE = {'tol_parm': 200}

# largest errors seen per group (printed at the end of the module with `pytest -s`)
OBSERVED = {}


def _note(group, key, value):
    g = OBSERVED.setdefault(group, {})
    g[key] = max(g.get(key, 0.0), float(value))


@pytest.fixture(scope='module', autouse=True)
def _report_observed():
    yield
    for group in sorted(OBSERVED):
        print('\nobserved maxima %s: %s' % (group, ', '.join('%s %.3e' % kv for kv in sorted(OBSERVED[group].items()))))


# ---- reference ----------------------------------------------------------------------------------------------------

def zmax(topo):
    """Upper end of k_pair4's Ewald fit in (alpha r)^2 units, as bl_create computes it."""
    return 1.02 * topo['ewald_alpha'] ** 2 * topo['cutoff'] ** 2


def fit_regime(topo):
    z = zmax(topo)
    return 10 if z <= ZMAX_DEG10 else (12 if z <= ZMAX_FIT_TOP else 'erfc')


class Reference(object):
    """Energy, forces and engine-named energy terms of one flattened system in float64, memoised on the coordinates
    and lambdas (several tests and switches evaluate the same walker coordinates)."""

    def __init__(self, topo):
        self.topo = topo
        self._memo = {}
        if topo['n_atoms'] > C_ORACLE_ABOVE:
            from oracle.c_oracle import COracle
            self._c, self._ff = COracle(topo), None
        else:
            from oracle.ncmc_oracle import ForceField
            self._c, self._ff = None, ForceField(topo)

    def __call__(self, x, lam_s=1.0, lam_e=1.0):
        x = np.ascontiguousarray(x, np.float64)
        key = (x.tobytes(), float(lam_s), float(lam_e))
        if key not in self._memo:
            if self._c is not None:
                from blues_b200._native import ENERGY_TERMS
                E, F, t = self._c.energy_forces(x, lam_s, lam_e)
                terms = dict(zip(ENERGY_TERMS, t.tolist()))
            else:
                E, F, comp = self._ff.energy_forces(x, self.topo['box'], lam_s, lam_e)
                terms = {k: sum(comp.get(nm, 0.0) for nm in names) for k, names in ORACLE_TERMS.items()}
            self._memo[key] = (float(E), F, terms, cutoff_edge_atoms(self.topo, x))
        return self._memo[key]


def cutoff_edge_atoms(topo, x):
    """Atoms of the pairs whose float64 distance lies within EDGE of the cutoff.  Float32 coordinates may put such a
    pair on either side, and the hard cutoff makes its force (~1 kJ/mol/nm for water, 1e-3 of a typical atom's force)
    all or nothing: the same edge rule as test_neighbour_and_exclusion_sets_bit_exact.  At random coordinates of
    wat_divaline about one pair in 5e5 lands there."""
    if topo['nb_method'] == 0:
        return np.zeros(0, np.int64)
    from scipy.spatial import cKDTree
    box, rc = np.asarray(topo['box'], float), float(topo['cutoff'])
    y = x - box * np.floor(x / box)
    y = np.where(y >= box, y - box, y)
    p = cKDTree(y, boxsize=box).query_pairs(rc + EDGE, output_type='ndarray')
    d = y[p[:, 0]] - y[p[:, 1]]
    d -= box * np.round(d / box)
    return np.unique(p[np.abs(np.linalg.norm(d, axis=1) - rc) < EDGE])


@pytest.fixture(scope='module')
def case():
    """case(name, alchemical=False, **createSystem overrides) -> (topo, fixture coordinates in nm, Reference), built
    once per module."""
    cache = {}

    def get(name, alchemical=False, **kw):
        key = (name, alchemical, tuple(sorted((k, str(v)) for k, v in kw.items())))
        if key not in cache:
            s, system, topo, x = load_case(name, alchemical, **kw)
            if name in MINIMIZE:
                from blues_b200 import _native
                eng = _native.Engine(topo, n_replicas=1, seed=1)
                eng.set_langevin_integrator(300.0, 1.0, 0.002)
                eng.set_positions(x)
                eng.minimize(MINIMIZE[name], 10.0)
                x = eng.get_positions(0)
                eng.close()
            cache[key] = (topo, x, Reference(topo))
        return cache[key]
    return get


def walker_sets(x0, R, scale=0.01):
    """R coordinate sets: the fixture plus a seeded displacement of about `scale` nm per atom (walker r: seed r)."""
    return [x0 + scale / np.sqrt(3.0) * np.random.RandomState(100 + r).standard_normal(x0.shape) for r in range(R)]


# ---- engine side --------------------------------------------------------------------------------------------------

def md_engine(topo, sets, seed=11, temperature=300.0):
    from blues_b200 import _native
    eng = _native.Engine(topo, n_replicas=len(sets), seed=seed)
    eng.set_langevin_integrator(temperature, 1.0, 0.002)
    for r, x in enumerate(sets):
        eng.set_positions(x, replica=r)
    eng.set_velocities(np.zeros_like(sets[0]))
    return eng


def capture(eng, steps=1):
    """md_run(steps), then per walker: positions, force-only forces (the last evaluation of md_run), energy-path forces
    (re-evaluated by get_energy at the same positions), potential energy and energy terms."""
    R = eng.n_replicas
    eng.md_run(steps)
    xs = [eng.get_positions(r) for r in range(R)]
    fast = [eng.get_forces(r) for r in range(R)]
    ep = eng.get_energy()[0]
    slow = [eng.get_forces(r) for r in range(R)]
    terms = [eng.get_energy_terms(r) for r in range(R)]
    return [dict(x=xs[r], f_fast=fast[r], f_energy=slow[r], energy=float(ep[r]), terms=terms[r]) for r in range(R)]


def energy_path(eng):
    """Energy-path evaluation at the coordinates already set: per walker positions, forces, energy and terms."""
    R = eng.n_replicas
    ep = eng.get_energy()[0]
    return [dict(x=eng.get_positions(r), f_energy=eng.get_forces(r), energy=float(ep[r]), terms=eng.get_energy_terms(r))
            for r in range(R)]


def check_walker(ref, w, group, label, lam=(1.0, 1.0), terms=True, alch_terms=False):
    """Forces of both paths against the oracle (and against each other), the energy and the terms."""
    E, F, T, edge = ref(w['x'], *lam)
    keep = np.ones(len(F), bool)
    keep[edge] = False
    _note(group, 'cutoff_edge_atoms', len(edge))
    errs = {'energy_path': rel_force_error(w['f_energy'][keep], F[keep])}
    if 'f_fast' in w:
        errs['force_only'] = rel_force_error(w['f_fast'][keep], F[keep])
        errs['force_only_vs_energy_path'] = rel_force_error(w['f_fast'][keep], w['f_energy'][keep])
    msg = '%s: %s (%d cutoff-edge atoms left out)' % (
        label, ', '.join('%s max rel %.3e rms rel %.3e' % (k, a, b) for k, (a, b) in sorted(errs.items())), len(edge))
    for k, (fmax, frms) in errs.items():
        _note(group, k + '_max_rel', fmax)
    assert all(fmax < FORCE_TOL for fmax, frms in errs.values()), msg
    erel = abs(w['energy'] - E) / max(abs(E), 1.0)
    _note(group, 'energy_rel', erel)
    assert erel < ENERGY_TOL, '%s energy %.6f oracle %.6f rel %.3e' % (label, w['energy'], E, erel)
    if terms:
        for k, b in T.items():
            a = w['terms'][k]
            assert abs(a - b) <= 1e-5 * max(abs(b), 1.0) + 1e-3, (label, k, a, b)
    if alch_terms:
        for k in ALCH_TERMS:
            a, b = w['terms'][k], T[k]
            _note(group, 'alch_term_abs', abs(a - b))
            assert abs(a - b) <= 1e-6 * max(abs(b), 1.0) + 1e-5, (label, k, a, b)


def check_md_walkers(topo, ref, R, group, label, steps=1, seed=11):
    """B-style check: R walkers at displaced fixture coordinates, `steps` MD steps, every walker against the oracle."""
    eng = md_engine(topo, walker_sets(ref.x0, R), seed=seed)
    try:
        ws = capture(eng, steps)
    finally:
        eng.close()
    for r, w in enumerate(ws):
        check_walker(ref, w, group, '%s walker %d/%d' % (label, r, R))
    if R > 1:
        assert not np.array_equal(ws[0]['x'], ws[1]['x'])
    return ws


def alchemical_walkers(topo, sets, lam_index, nsteps=10):
    from blues_b200 import _native
    ls, le = lambda_tables(nsteps)
    eng = _native.Engine(topo, n_replicas=len(sets), seed=1)
    try:
        eng.set_ncmc_integrator(300.0, 1.0, 0.002, 'H V R O R V H', nsteps, 1, 0.2, 0.8, ls, le)
        eng.set_global('lambda_step', lam_index)
        for r, x in enumerate(sets):
            eng.set_positions(x, replica=r)
        return energy_path(eng), (ls[lam_index], le[lam_index])
    finally:
        eng.close()


def _with_x0(get, name, alchemical=False, **kw):
    topo, x0, ref = get(name, alchemical, **kw)
    ref.x0 = x0
    return topo, ref


# ---- A. force-only path against the oracle -----------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize('name', ['wat_divaline', 'tol_parm', 't4l_surrogate', 'vac_divaline'])
def test_force_only_and_energy_path_forces_match_oracle(name, case):
    """k_pair4 at Ewald-fit degree 10 (wat_divaline, t4l_surrogate) and 12 (tol_parm); k_pair2<NoCutoff, false>
    (vac_divaline); force-only reciprocal space."""
    topo, ref = _with_x0(case, name)
    eng = md_engine(topo, [ref.x0])
    try:
        w = capture(eng)[0]
    finally:
        eng.close()
    check_walker(ref, w, 'A', name)


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['wat_divaline', 'tol_parm'])
def test_force_only_path_really_runs_the_packed_kernel(name, case, monkeypatch):
    """The same run with k_pair4 switched off (BLUES_B200_PAIR_X2=0: k_pair2 on the force-only path): the force-only
    forces must differ in at least one bit (another kernel with another Ewald fit ran), and both be within tolerance.
    Same seed and start, so every other launch is identical."""
    topo, ref = _with_x0(case, name)
    out = {}
    for flag in (None, '0'):
        if flag is None:
            monkeypatch.delenv('BLUES_B200_PAIR_X2', raising=False)
        else:
            monkeypatch.setenv('BLUES_B200_PAIR_X2', flag)
        eng = md_engine(topo, [ref.x0], seed=5)
        try:
            out[flag] = capture(eng)[0]
        finally:
            eng.close()
        check_walker(ref, out[flag], 'A', '%s PAIR_X2=%s' % (name, flag or 'default'))
    assert not np.array_equal(out[None]['f_fast'], out['0']['f_fast'])


# ---- B. many walkers, each at its own coordinates ----------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize('name,R', [(n, R) for n in ('wat_divaline', 'tol_parm') for R in (1, 2, 3, 8)] +
                         [('t4l_surrogate', 3)])
def test_every_walker_matches_oracle_at_its_own_coordinates(name, R, case):
    """R > 2 takes k_pme_spread<256> with 4 y-bands, k_pme_gather and the many-walker builder configuration."""
    topo, ref = _with_x0(case, name)
    check_md_walkers(topo, ref, R, 'B', name)


@pytest.mark.gpu
@pytest.mark.parametrize('R', [3, 8])
@pytest.mark.parametrize('lam_index', [0, 7, 15])
def test_alchemical_walkers_match_oracle_at_their_own_coordinates(R, lam_index, case):
    """Energy path (k_alch has no force-only variant): per walker forces, energy and the three alchemical terms."""
    topo, ref = _with_x0(case, 'wat_divaline', True)
    ws, lam = alchemical_walkers(topo, walker_sets(ref.x0, R), lam_index)
    for r, w in enumerate(ws):
        check_walker(ref, w, 'B', 'alchemical lambda_step %d walker %d/%d' % (lam_index, r, R), lam=lam, terms=False,
                     alch_terms=True)


@pytest.mark.gpu
@pytest.mark.parametrize('name,R', [('wat_divaline', 3), ('tol_parm', 8)])
def test_walker_slot_does_not_change_a_bit(name, R, case):
    """The coordinate sets rotated across the slots of one engine (slot r gets set r + 1 mod R) give the same positions
    after a step, force-only forces, energy-path forces, energies and terms bit for bit: the charge spread, the force and
    energy accumulators are integers, and the batched FFTs transform every walker's grid alike.  At 0 K the step adds
    no noise, so the walker's state does not depend on its slot's noise stream."""
    topo, ref = _with_x0(case, name)
    sets = walker_sets(ref.x0, R)
    eng = md_engine(topo, sets, temperature=0.0)
    try:
        a = capture(eng)
        for r in range(R):
            eng.set_positions(sets[(r + 1) % R], replica=r)
        eng.set_velocities(np.zeros_like(sets[0]))
        b = capture(eng)
    finally:
        eng.close()
    for r in range(R):
        s = (r + 1) % R
        for k in ('x', 'f_fast', 'f_energy'):
            assert np.array_equal(b[r][k], a[s][k]), (k, r, s, float(np.max(np.abs(b[r][k] - a[s][k]))))
        assert b[r]['energy'] == a[s]['energy'] and b[r]['terms'] == a[s]['terms'], (r, s)
    assert not np.array_equal(a[0]['f_fast'], a[1]['f_fast'])


# ---- C. Ewald-fit regimes and the cutoff edge --------------------------------------------------------------------

SYN_BOX = np.array([2.0, 2.2, 2.4])
SYN_CUTOFF = 0.9
SYN_SKIN = 0.14 * SYN_CUTOFF          # the engine's default Verlet skin
# ewaldErrorTolerance -> zmax = 1.02 ln(1 / (2 tol)): 4.6, 4.9, 7.0, 10.9, 12.3
REGIMES = [(5.5e-3, 4.6, 10), (4.1e-3, 4.9, 12), (5.2e-4, 7.0, 12), (1.14e-5, 10.9, 12), (2.9e-6, 12.3, 'erfc')]
SMALL_GRID = (9, 10, 12)


def synthetic_system(tol=5e-4, grid=None):
    """200 charged Lennard-Jones particles in a 2.0 x 2.2 x 2.4 nm box, r_c 0.9 nm: 100 dimers (partners 0.1-0.3 nm
    apart, not excluded) on a jittered 4 x 5 x 5 lattice, no two other atoms closer than 0.15 nm.  At this density
    hundreds of pairs fall in each of [0.97 r_c, r_c), (r_c, 1.01 r_c] and (1.01 r_c, r_c + skin).
    grid: (nx, ny, nz) overrides the PME grid (alpha still from `tol`)."""
    from blues_b200.system import System, NonbondedForce, PME, pme_parameters
    rng = np.random.RandomState(7)
    lattice = np.stack(np.meshgrid(np.arange(4), np.arange(5), np.arange(5), indexing='ij'), -1).reshape(-1, 3)
    centres = (lattice + 0.5 + 0.15 * (rng.rand(len(lattice), 3) - 0.5)) * SYN_BOX / np.array([4, 5, 5])
    x = []
    for c in centres:
        while True:
            d = rng.uniform(0.1, 0.3)
            v = rng.standard_normal(3)
            pair = [c + 0.5 * d * v / np.linalg.norm(v), c - 0.5 * d * v / np.linalg.norm(v)]
            if not x:
                break
            dd = np.asarray(x)[:, None, :] - np.asarray(pair)[None, :, :]
            dd -= SYN_BOX * np.round(dd / SYN_BOX)
            if np.min(np.linalg.norm(dd, axis=2)) >= 0.15:
                break
        x.extend(pair)
    x = np.asarray(x) % SYN_BOX
    n = len(x)
    s = System(n)
    s.masses = rng.uniform(12.0, 40.0, n)
    s.box = SYN_BOX.copy()
    nb = NonbondedForce(n)
    s.addForce(nb)
    q = rng.uniform(0.2, 0.6, n // 2)
    nb.charge[:] = np.stack([q, -q], 1).reshape(-1)
    nb.sigma[:] = rng.uniform(0.10, 0.16, n)
    nb.epsilon[:] = rng.uniform(0.1, 0.5, n)
    nb.method = PME
    nb.cutoff = SYN_CUTOFF
    nb.setEwaldErrorTolerance(tol)
    if grid is not None:
        nb.pme_params = (pme_parameters(SYN_CUTOFF, tol, SYN_BOX)[0],) + tuple(grid)
    return s.flatten(), x


def pair_distances(x, box):
    i, j = np.triu_indices(len(x), 1)
    d = x[i] - x[j]
    d -= box * np.round(d / box)
    return np.linalg.norm(d, axis=1)


def test_synthetic_cases_land_in_their_intended_ewald_fit_regime():
    """CPU: the ewaldErrorTolerance of each GPU case below puts zmax where the case means it to be (a change of the
    PME parameter rule must not move them silently), and the coordinates populate every distance range."""
    for tol, target, regime in REGIMES:
        topo, x = synthetic_system(tol)
        assert abs(zmax(topo) - target) < 0.05, (tol, zmax(topo), target)
        assert fit_regime(topo) == regime, (tol, zmax(topo), regime)
    assert abs(zmax(synthetic_system(REGIMES[1][0])[0]) - ZMAX_DEG10) < 0.15          # just past the degree switch
    assert abs(zmax(synthetic_system(REGIMES[3][0])[0]) - ZMAX_FIT_TOP) < 0.7         # near the top of the fit
    topo, x = synthetic_system(5e-4, SMALL_GRID)
    assert tuple(topo['pme_grid']) == SMALL_GRID
    assert topo['n_atoms'] == 200 and abs(np.sum(topo['charge'])) < 1e-12
    r = pair_distances(x, SYN_BOX)
    rc = SYN_CUTOFF
    assert np.min(r) >= 0.1 - 1e-12
    for lo, hi in ((0.1, 0.3), (0.97 * rc, rc), (rc, 1.01 * rc), (1.01 * rc, rc + SYN_SKIN)):
        assert np.count_nonzero((r > lo) & (r < hi)) >= 50, (lo, hi)


@pytest.fixture(scope='module')
def synthetic():
    cache = {}

    def get(tol=5e-4, grid=None):
        key = (tol, grid)
        if key not in cache:
            topo, x = synthetic_system(tol, grid)
            ref = Reference(topo)
            ref.x0 = x
            cache[key] = (topo, ref)
        return cache[key]
    return get


@pytest.mark.gpu
@pytest.mark.parametrize('tol,target,regime', REGIMES, ids=['zmax%.1f' % z for _, z, _ in REGIMES])
def test_ewald_fit_regimes_and_cutoff_edge_match_oracle(tol, target, regime, synthetic):
    """Both paths and the energy at each regime of the fit; pairs between r_c and r_c + skin are in the list and must
    contribute nothing."""
    topo, ref = synthetic(tol)
    check_md_walkers(topo, ref, 1, 'C', 'zmax %.1f' % target)


@pytest.mark.gpu
@pytest.mark.parametrize('R', [1, 3])
def test_small_odd_pme_grid_matches_oracle(R, synthetic):
    """9 x 10 x 12 grid: the order-5 stencil covers most of a plane, the spread takes whole cell rows."""
    topo, ref = synthetic(5e-4, SMALL_GRID)
    check_md_walkers(topo, ref, R, 'C', 'grid 9x10x12')


# ---- D. reaction field (CutoffPeriodic) --------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize('R', [1, 3])
def test_reaction_field_walkers_match_oracle(R, case):
    topo, ref = _with_x0(case, 'wat_divaline', **RF)
    assert topo['nb_method'] == 2
    check_md_walkers(topo, ref, R, 'D', 'reaction field')


@pytest.mark.gpu
@pytest.mark.parametrize('lam_index', [0, 7, 15])
def test_reaction_field_alchemical_walkers_match_oracle(lam_index, case):
    topo, ref = _with_x0(case, 'wat_divaline', True, **RF)
    ws, lam = alchemical_walkers(topo, walker_sets(ref.x0, 3), lam_index)
    for r, w in enumerate(ws):
        check_walker(ref, w, 'D', 'reaction field alchemical lambda_step %d walker %d' % (lam_index, r), lam=lam,
                     alch_terms=True)


@pytest.mark.gpu
@pytest.mark.parametrize('R', [1, 3])
def test_reaction_field_neighbour_and_exclusion_sets(R, case):
    """Same edge rule as test_neighbour_and_exclusion_sets_bit_exact: a pair may differ only within float32 rounding
    of the cutoff."""
    from blues_b200 import _native
    topo, ref = _with_x0(case, 'wat_divaline', **RF)
    sets = walker_sets(ref.x0, R)
    eng = _native.Engine(topo, n_replicas=R, seed=1)
    try:
        eng.set_langevin_integrator(300.0, 1.0, 0.002)
        for r, x in enumerate(sets):
            eng.set_positions(x, replica=r)
        codes = [eng.neighbor_pairs(r) for r in range(R)]
    finally:
        eng.close()
    from oracle.ncmc_oracle import ForceField
    ff = ForceField(topo)
    n = topo['n_atoms']
    for r in range(R):
        want = ff.neighbor_pairs(sets[r], topo['box'])
        assert len(codes[r]) == len(np.unique(codes[r]))
        diff = np.concatenate([np.setdiff1d(codes[r], want), np.setdiff1d(want, codes[r])])
        if len(diff):
            d = sets[r][diff // n] - sets[r][diff % n]
            d -= topo['box'] * np.round(d / topo['box'])
            edge = float(np.max(np.abs(np.linalg.norm(d, axis=1) - topo['cutoff'])))
            assert edge < 5e-7, (r, len(diff), edge)


# ---- E. run-time kernel switches ---------------------------------------------------------------------------------

SWITCHES = ([('PAIR_X2', v) for v in ('0', '4')] + [('PAIR_LANES', v) for v in ('4', '16', '32')] +
            [('ZFINE', '1'), ('INT_BLOCK', '64'), ('FOLD_ZERO', '0'), ('GRAPH_STEPS', '1'), ('PDL', '0'),
             ('SKIN', '0.05'), ('BUILD_CQ', '16'), ('BUILD_PER_SM', '1'), ('PAIR_PER_SM', '1'), ('SPREAD_THREADS', '512'),
             ('NO_PRIORITY', '1')])
SWITCH_CASES = ([(var, val, 'wat_divaline', (1, 3)) for var, val in SWITCHES] +
                [('PAIR_SPLIT', '1', 'wat_divaline', (8,))] +
                [(var, val, 'small_grid', (1, 3)) for var, val in (('SPREAD_SPLIT', '2'), ('SPREAD_THREADS', '512'))])


@pytest.mark.gpu
@pytest.mark.parametrize('var,val,name,Rs', SWITCH_CASES,
                         ids=['%s=%s-%s' % (v, x, n) for v, x, n, _ in SWITCH_CASES])
def test_kernel_switch_keeps_every_walker_on_the_oracle(var, val, name, Rs, case, synthetic, monkeypatch):
    """tools/README.md: no run-time switch changes a result beyond float summation order.  Three MD steps, so that the
    last force-only evaluation runs on lists that were not rebuilt in it (PAIR_SPLIT: the walkers beside the builder).
    GRAPH_STEPS only batches NCMC steps: that switch is also checked on an NCMC run, which must be bitwise the
    default's."""
    monkeypatch.setenv('BLUES_B200_' + var, val)
    if name == 'small_grid':
        topo, ref = synthetic(5e-4, SMALL_GRID)
    else:
        topo, ref = _with_x0(case, name)
    for R in Rs:
        check_md_walkers(topo, ref, R, 'E', '%s=%s %s' % (var, val, name), steps=3)
    if var == 'GRAPH_STEPS':
        atopo, aref = _with_x0(case, name, True)
        runs = []
        for flag in (val, None):
            if flag is None:
                monkeypatch.delenv('BLUES_B200_' + var)
            runs.append(_ncmc_run(atopo, aref.x0, 9))
        assert np.array_equal(runs[0][0], runs[1][0]) and runs[0][1] == runs[1][1]


def _ncmc_run(topo, x, steps, nsteps=20):
    from blues_b200 import _native
    ls, le = lambda_tables(nsteps)
    eng = _native.Engine(topo, n_replicas=2, seed=3)
    try:
        eng.set_ncmc_integrator(300.0, 1.0, 0.002, 'H V R O R V H', nsteps, 1, 0.2, 0.8, ls, le)
        eng.set_positions(x)
        eng.velocities_to_temperature(300.0)
        eng.ncmc_run(steps)
        return eng.get_positions(1), eng.get_global('protocol_work', 1)
    finally:
        eng.close()
