"""Generate the committed fixtures under tests/golden/ from the reference's data files.

Run with ``BLUES_REFERENCE_DATA`` naming ``blues/tests/data`` of a MobleyLab/blues checkout:

    BLUES_REFERENCE_DATA=<checkout>/blues/tests/data python tests/golden/make_fixtures.py [--reference-tests | --spread-lambda]

Outputs
  tol_parm.npz / wat_divaline.npz / vac_divaline.npz
      Structure arrays parsed from ``blues/tests/data/*.prmtop`` + ``.inpcrd`` (complete AMBER fixtures).
  t4l_surrogate.npz
      T4 lysozyme L99A + toluene at the reference's coordinates (``eqToluene.inpcrd``/``.pdb``, 22 340 atoms).
      ``eqToluene.prmtop`` is missing from the reference checkout (``.MISSING_LARGE_BLOBS``), so the force field
      is a SURROGATE: real geometry/box/composition, TIP3P water, toluene parameters transplanted from
      ``TOL-parm.prmtop``, AMBER-like per-element Lennard-Jones and template charges for the protein,
      structure-based bonded equilibrium values.  Valid as a throughput workload with the right N, density,
      constraint topology and PME grid — NOT a physical model of T4L.
  oracle_vectors.npz
      Energies (by term) and forces of the float64 oracle on those systems, for the CPU-side golden tests.
  spread_lambda_protocol.json (--spread-lambda)
      utils.spreadLambdaProtocol tables for the cases of tests/test_host_logic.py; its ``source`` entry says which
      function computed them (the reference's, executed from its source text, or this package's).
"""
import os
import sys
import math
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = os.environ.get('BLUES_REFERENCE_DATA')

from blues_b200.structure import Structure, load_file, load_pdb, read_inpcrd  # noqa: E402
from blues_b200 import unit as u  # noqa: E402


def graph_distances(adj, start):
    dist = {start: 0}
    frontier = [start]
    while frontier:
        nxt = []
        for a in frontier:
            for b in adj[a]:
                if b not in dist:
                    dist[b] = dist[a] + 1
                    nxt.append(b)
        frontier = nxt
    return dist


def toluene_classes(z, bonds, n):
    """class of each toluene atom = (element, graph distance from the methyl carbon)"""
    adj = [[] for _ in range(n)]
    for i, j in bonds:
        adj[i].append(j)
        adj[j].append(i)
    methyl = [a for a in range(n) if z[a] == 6 and sum(1 for b in adj[a] if z[b] == 1) == 3][0]
    dist = graph_distances(adj, methyl)
    return [(int(z[a]), dist[a]) for a in range(n)], adj


# AMBER-like Lennard-Jones (sigma Å, eps kcal/mol) by simple chemical class
LJ = {'CT': (3.39967, 0.1094), 'C': (3.39967, 0.0860), 'N': (3.25000, 0.1700), 'O': (2.95992, 0.2100),
      'OH': (3.06647, 0.2104), 'S': (3.56359, 0.2500), 'H': (1.06908, 0.0157), 'HC': (2.64953, 0.0157),
      'H1': (2.47135, 0.0157), 'HA': (2.59964, 0.0150), 'HO': (0.0, 0.0), 'HP': (1.95998, 0.0157),
      'OW': (3.15075, 0.1521), 'HW': (0.0, 0.0), 'Cl-': (4.47766, 0.0356)}
BACKBONE_Q = {'N': -0.4157, 'H': 0.2719, 'CA': 0.0337, 'HA': 0.0823, 'C': 0.5973, 'O': -0.5679}
FORMAL = {'LYS': 1, 'ARG': 1, 'ASP': -1, 'GLU': -1, 'HIP': 1}
COV = {1: 0.31, 6: 0.76, 7: 0.71, 8: 0.66, 16: 1.05}


def build_t4l_surrogate():
    pdb = load_pdb(os.path.join(REF, 'eqToluene.pdb'))
    xyz, _, box = read_inpcrd(os.path.join(REF, 'eqToluene.inpcrd'))
    tol = load_file(os.path.join(REF, 'TOL-parm.prmtop'), xyz=os.path.join(REF, 'TOL-parm.inpcrd'))
    n = pdb.n_atoms
    z = pdb.atomic_numbers.copy()
    names = pdb.atom_names
    rp = pdb.residue_pointers
    rnames = pdb.residue_names
    nres = len(rnames)
    protein_res = [r for r in range(nres) if rnames[r] not in ('LIG', 'HOH', 'WAT', 'Cl-', 'CL', 'Na+')]
    from scipy.spatial import cKDTree

    bonds = set()
    # protein: distance perception within a residue and across the peptide bond
    prot_atoms = np.concatenate([np.arange(rp[r], rp[r + 1]) for r in protein_res])
    tree = cKDTree(xyz[prot_atoms])
    for a, b in tree.query_pairs(2.2):
        i, j = int(prot_atoms[a]), int(prot_atoms[b])
        if z[i] == 1 and z[j] == 1:
            continue
        ri, rj = pdb.atom_residue[i], pdb.atom_residue[j]
        if abs(ri - rj) > 1:
            if not (names[i] == 'SG' and names[j] == 'SG'):
                continue
        if ri != rj and not ({names[i], names[j]} == {'C', 'N'}):
            continue
        d = np.linalg.norm(xyz[i] - xyz[j])
        if d < 1.25 * (COV[int(z[i])] + COV[int(z[j])]):
            bonds.add((min(i, j), max(i, j)))
    # each hydrogen keeps only its closest heavy partner
    adj = {}
    for i, j in bonds:
        adj.setdefault(i, []).append(j)
        adj.setdefault(j, []).append(i)
    for a in prot_atoms:
        a = int(a)
        if z[a] == 1 and len(adj.get(a, [])) > 1:
            best = min(adj[a], key=lambda b: np.linalg.norm(xyz[a] - xyz[b]))
            for b in adj[a]:
                if b != best:
                    bonds.discard((min(a, b), max(a, b)))
    # ligand from CONECT, waters O-H
    for i, j in pdb.bonds:
        bonds.add((int(min(i, j)), int(max(i, j))))
    waters = []
    for r in range(nres):
        if rnames[r] in ('HOH', 'WAT'):
            a0 = rp[r]
            o = a0 + int(np.argmax(z[a0:a0 + 3] == 8))
            hs = [a for a in range(a0, a0 + 3) if a != o]
            waters.append((o, hs[0], hs[1]))
            bonds.add((min(o, hs[0]), max(o, hs[0])))
            bonds.add((min(o, hs[1]), max(o, hs[1])))
    bonds = np.asarray(sorted(bonds), int)
    adj = [[] for _ in range(n)]
    for i, j in bonds:
        adj[i].append(int(j))
        adj[j].append(int(i))
    water_atoms = set(a for w in waters for a in w)

    # ---- atom classes, LJ, charges ---------------------------------------------------------------------
    sigma = np.zeros(n)
    eps = np.zeros(n)
    q = np.zeros(n)
    types = [''] * n
    sp2 = np.zeros(n, bool)
    for a in range(n):
        za, nb = int(z[a]), adj[a]
        if za == 6:
            sp2[a] = len(nb) <= 3
        elif za == 7:
            sp2[a] = len(nb) <= 3
        elif za == 8:
            sp2[a] = len(nb) == 1
    lig = list(range(rp[rnames.index('LIG')], rp[rnames.index('LIG') + 1]))
    for a in range(n):
        za, nb = int(z[a]), adj[a]
        rn = rnames[pdb.atom_residue[a]]
        if a in water_atoms:
            t = 'OW' if za == 8 else 'HW'
        elif rn in ('Cl-', 'CL'):
            t = 'Cl-'
        elif za == 6:
            t = 'C' if sp2[a] else 'CT'
        elif za == 7:
            t = 'N'
        elif za == 8:
            t = 'O' if len(nb) == 1 else 'OH'
        elif za == 16:
            t = 'S'
        elif za == 1:
            p = nb[0] if nb else -1
            zp = int(z[p]) if p >= 0 else 6
            if zp == 7:
                t = 'H'
            elif zp in (8, 16):
                t = 'HO'
            elif zp == 6 and sp2[p]:
                t = 'HA'
            elif zp == 6:
                ewd = sum(1 for b in adj[p] if z[b] in (7, 8, 16))
                t = 'H1' if ewd == 1 else ('HP' if ewd > 1 else 'HC')
            else:
                t = 'HC'
        else:
            t = 'CT'
        types[a] = t
        sigma[a], eps[a] = LJ[t]
    # water / ion charges
    for (o, h1, h2) in waters:
        q[o], q[h1], q[h2] = -0.834, 0.417, 0.417
    for a in range(n):
        if types[a] == 'Cl-':
            q[a] = -1.0
    # protein charges: backbone template + generic polar groups, then shift each residue to its formal charge
    for r in protein_res:
        atoms = list(range(rp[r], rp[r + 1]))
        for a in atoms:
            nm = names[a]
            if nm in BACKBONE_Q:
                q[a] = BACKBONE_Q[nm]
            elif z[a] == 1 and adj[a] and z[adj[a][0]] in (7, 8, 16):
                q[a] = 0.40
            elif z[a] in (7, 8, 16):
                q[a] = -0.40 * max(1, sum(1 for b in adj[a] if z[b] == 1)) if any(z[b] == 1 for b in adj[a]) else -0.50
            elif z[a] == 6 and any(z[b] in (7, 8) for b in adj[a]) and names[a] not in ('CA', 'C'):
                q[a] = 0.25
            elif z[a] == 1:
                q[a] = 0.05
            else:
                q[a] = -0.10
        formal = FORMAL.get(rnames[r], 0)
        if r == protein_res[0]:
            formal += 1
        if 'OXT' in [names[a] for a in atoms]:
            formal -= 1
        q[atoms] += (formal - q[atoms].sum()) / len(atoms)
    # toluene: transplant charges / LJ by (element, distance from the methyl carbon)
    tcls, _ = toluene_classes(tol.atomic_numbers[:15], [tuple(b) for b in tol.bonds if b[0] < 15 and b[1] < 15], 15)
    lig_local = {a: k for k, a in enumerate(lig)}
    lcls, _ = toluene_classes(z[lig], [(lig_local[i], lig_local[j]) for i, j in bonds if i in lig_local and j in lig_local], len(lig))
    for k, a in enumerate(lig):
        same = [m for m in range(15) if tcls[m] == lcls[k]]
        q[a] = float(np.mean(tol.charges[same]))
        sigma[a] = float(tol.lj_sigma[same[0]])
        eps[a] = float(tol.lj_epsilon[same[0]])
        types[a] = tol.atom_types[same[0]]
    q[lig] -= q[lig].sum() / len(lig)
    total = q.sum()
    q[prot_atoms] -= total / len(prot_atoms)     # neutralise the tiny remainder

    # ---- bonded terms (equilibrium values from the structure itself) ------------------------------------
    bl = np.linalg.norm(xyz[bonds[:, 0]] - xyz[bonds[:, 1]], axis=1)
    bk = np.where((z[bonds[:, 0]] == 1) | (z[bonds[:, 1]] == 1), 340.0, 310.0)
    for k, (i, j) in enumerate(bonds):
        if i in water_atoms:
            bl[k], bk[k] = 0.9572, 553.0
    angles, ak, at0 = [], [], []
    for b in range(n):
        nb = adj[b]
        for x in range(len(nb)):
            for y in range(x + 1, len(nb)):
                a, c = nb[x], nb[y]
                v1, v2 = xyz[a] - xyz[b], xyz[c] - xyz[b]
                th = math.acos(np.clip(np.dot(v1, v2) / np.linalg.norm(v1) / np.linalg.norm(v2), -1, 1))
                if b in water_atoms:
                    th, k_ = math.radians(104.52), 100.0
                elif z[a] == 1 and z[c] == 1:
                    k_ = 35.0
                elif z[a] == 1 or z[c] == 1:
                    k_ = 50.0
                else:
                    k_ = 63.0
                angles.append((a, b, c))
                ak.append(k_)
                at0.append(th)
    dih, dk, dn, dph, dig = [], [], [], [], []
    seen14 = set()
    bonded13 = set()
    for b in range(n):
        for a in adj[b]:
            bonded13.add((min(a, b), max(a, b)))
            for c in adj[b]:
                if c != a:
                    bonded13.add((min(a, c), max(a, c)))
    for b, c in bonds:
        if b in water_atoms:
            continue
        for a in adj[b]:
            if a == c:
                continue
            for d_ in adj[c]:
                if d_ == b or d_ == a:
                    continue
                key = (min(a, d_), max(a, d_))
                ignore = key in seen14 or key in bonded13
                seen14.add(key)
                if sp2[b] and sp2[c]:
                    k_, n_, ph = 2.5, 2, math.pi
                else:
                    k_, n_, ph = 0.156, 3, 0.0
                dih.append((a, int(b), int(c), d_))
                dk.append(k_)
                dn.append(n_)
                dph.append(ph)
                dig.append(ignore)

    s = Structure()
    s.n_atoms = n
    s.atom_names = list(names)
    s.atom_types = types
    s.atomic_numbers = z
    s.masses = pdb.masses.copy()
    s.charges = q
    s.lj_sigma, s.lj_epsilon = sigma, eps
    s.residue_names = list(rnames)
    s.residue_pointers = rp.copy()
    s.atom_residue = pdb.atom_residue.copy()
    s.bonds, s.bond_k, s.bond_r0 = bonds, bk, bl
    s.angles = np.asarray(angles, int).reshape(-1, 3)
    s.angle_k, s.angle_t0 = np.asarray(ak), np.asarray(at0)
    s.dihedrals = np.asarray(dih, int).reshape(-1, 4)
    s.dihedral_k, s.dihedral_per, s.dihedral_phase = np.asarray(dk), np.asarray(dn, float), np.asarray(dph)
    s.dihedral_scee = np.full(len(dih), 1.2)
    s.dihedral_scnb = np.full(len(dih), 2.0)
    s.dihedral_ignore_end = np.asarray(dig, bool)
    s.dihedral_improper = np.zeros(len(dih), bool)
    s.coordinates = xyz.copy()
    s.box = list(box)
    return s


def oracle_vectors(structs):
    from oracle.ncmc_oracle import ForceField
    from blues_b200.alchemy import AbsoluteAlchemicalFactory, AlchemicalRegion
    out = {}
    cases = [('tol_parm', dict(nonbondedMethod='PME', nonbondedCutoff=8.0 * u.angstroms, constraints='HBonds'), list(range(15))),
             ('wat_divaline', dict(nonbondedMethod='PME', nonbondedCutoff=10.0 * u.angstroms, constraints='HBonds',
                                   ewaldErrorTolerance=0.005), list(range(16, 35))),
             ('vac_divaline', dict(nonbondedMethod='NoCutoff', constraints='HBonds'), list(range(16, 35)))]
    for name, kw, alch_atoms in cases:
        s = structs[name]
        system = s.createSystem(**kw)
        x = s.coordinates * 0.1
        t = system.flatten()
        E, F, comp = ForceField(t).energy_forces(x, t['box'])
        out[name + '/md/energy'] = E
        out[name + '/md/forces'] = F
        for k, v in comp.items():
            out[name + '/md/term/' + k] = v
        alch = AbsoluteAlchemicalFactory().create_alchemical_system(system, AlchemicalRegion(alchemical_atoms=alch_atoms))
        ta = alch.flatten()
        ffa = ForceField(ta)
        for ls, le in ((1.0, 1.0), (0.5, 0.25), (0.0, 0.0)):
            E, F, comp = ffa.energy_forces(x, ta['box'], ls, le)
            tag = '%s/alch_%g_%g' % (name, ls, le)
            out[tag + '/energy'] = E
            out[tag + '/forces'] = F
            for k, v in comp.items():
                out[tag + '/term/' + k] = v
    return out


def reference_bookkeeping():
    """Run the reference's own pure-Python bookkeeping functions (source extracted with ``ast`` from the reference
    checkout, executed with a stub logger) on a grid of inputs → golden table for calculateNCMCSteps
    (blues/utils.py:89-145) and _get_prop_lambda (blues/integrators.py:147-157)."""
    import ast
    import json
    import logging
    refroot = os.path.dirname(os.path.dirname(REF))

    def extract(path, name):
        src = open(path).read()
        tree = ast.parse(src)
        for node in ast.walk(tree):
            if isinstance(node, ast.FunctionDef) and node.name == name:
                return ast.get_source_segment(src, node)
        raise KeyError(name)

    ns = {'logger': logging.getLogger('ref'), 'sys': sys, 'floor': math.floor, 'ceil': math.ceil}
    logging.getLogger('ref').setLevel(logging.CRITICAL)
    exec(extract(os.path.join(refroot, 'utils.py'), 'calculateNCMCSteps'), ns)
    import textwrap
    exec(textwrap.dedent(extract(os.path.join(refroot, 'integrators.py'), '_get_prop_lambda')), ns)
    out = {'calculateNCMCSteps': [], 'get_prop_lambda': []}
    for nsteps in (2, 4, 10, 11, 20, 99, 100, 500, 1000, 1001, 2500, 5000, 10000):
        for nprop in (1, 2, 3, 5):
            for pl in (0.0, 0.1, 0.2, 0.3, 0.45, 0.5):
                res = ns['calculateNCMCSteps'](nstepsNC=nsteps, nprop=nprop, propLambda=pl)
                out['calculateNCMCSteps'].append([[nsteps, nprop, pl], res])
    for pl in (0.0, 0.05, 0.1, 0.2, 0.3, 0.33333, 0.45, 0.5, 0.6, -0.1):
        out['get_prop_lambda'].append([pl, list(ns['_get_prop_lambda'](None, pl))])
    with open(os.path.join(HERE, 'reference_bookkeeping.json'), 'w') as f:
        json.dump(out, f)
    print('reference bookkeeping rows:', len(out['calculateNCMCSteps']), len(out['get_prop_lambda']))


def ethylene_fixture():
    """blues/tests/data/ethylene_system.xml + ethylene_structure.pdb → ethylene.json (the reference's only known-answer
    system, tests/test_ethylene.py)."""
    import json
    import xml.etree.ElementTree as ET
    root = ET.parse(os.path.join(REF, 'ethylene_system.xml')).getroot()
    out = {'mass': [float(p.get('mass')) for p in root.find('Particles')],
           'constraints': [[int(c.get('p1')), int(c.get('p2')), float(c.get('d'))] for c in root.find('Constraints')]}
    for f in root.find('Forces'):
        t = f.get('type')
        if t == 'HarmonicBondForce':
            out['bonds'] = [[int(b.get('p1')), int(b.get('p2')), float(b.get('d')), float(b.get('k'))] for b in f.find('Bonds')]
        elif t == 'HarmonicAngleForce':
            out['angles'] = [[int(a.get('p1')), int(a.get('p2')), int(a.get('p3')), float(a.get('a')), float(a.get('k'))]
                             for a in f.find('Angles')]
        elif t == 'PeriodicTorsionForce':
            out['torsions'] = [[int(x.get('p1')), int(x.get('p2')), int(x.get('p3')), int(x.get('p4')),
                                int(x.get('periodicity')), float(x.get('phase')), float(x.get('k'))] for x in f.find('Torsions')]
        elif t == 'CustomNonbondedForce':
            out['custom_nonbonded'] = {'energy': f.get('energy'), 'method': int(f.get('method')),
                                       'params': [[float(p.get('param1')), float(p.get('param2')), float(p.get('param3'))]
                                                  for p in f.find('Particles')],
                                       'set1': [int(p.get('index')) for p in f.find('InteractionGroups')[0].find('Set1')],
                                       'set2': [int(p.get('index')) for p in f.find('InteractionGroups')[0].find('Set2')]}
        elif t == 'CustomCentroidBondForce':
            groups = [[int(p.get('p')) for p in g] for g in f.find('Groups')]
            out['centroid_bond'] = {'energy': f.get('energy'), 'groups': groups, 'k': float(f.find('Bonds')[0].get('param1'))}
    pdb = load_pdb(os.path.join(REF, 'ethylene_structure.pdb'))
    out['positions_nm'] = (pdb.coordinates * 0.1).tolist()
    out['atomic_numbers'] = pdb.atomic_numbers.tolist()
    out['residue_names'] = pdb.residue_names
    with open(os.path.join(HERE, 'ethylene.json'), 'w') as fh:
        json.dump(out, fh)
    print('ethylene fixture:', len(out['mass']), 'particles')


def reference_tests():
    """Verbatim copies of the reference's own test files and the data they read (tests/golden/reference_checkout/):
    fixtures of tests/test_gpu_reference_suite.py, which runs them unmodified against the CUDA engine on the GPU box."""
    import shutil
    root = os.path.dirname(os.path.dirname(REF))          # <checkout>/blues
    dst = os.path.join(HERE, 'reference_checkout', 'blues', 'tests')
    os.makedirs(os.path.join(dst, 'data'), exist_ok=True)
    for name in ('test_simulation.py', 'test_randomrotation.py', 'test_ethylene.py'):
        shutil.copyfile(os.path.join(root, 'tests', name), os.path.join(dst, name))
    for name in ('TOL-parm.prmtop', 'TOL-parm.inpcrd', 'ethylene_system.xml', 'ethylene_structure.pdb'):
        shutil.copyfile(os.path.join(REF, name), os.path.join(dst, 'data', name))
    import hashlib
    digests = {}
    for rel in ('test_simulation.py', 'test_randomrotation.py', 'test_ethylene.py', 'data/TOL-parm.prmtop',
                'data/TOL-parm.inpcrd', 'data/ethylene_system.xml', 'data/ethylene_structure.pdb'):
        with open(os.path.join(dst, rel), 'rb') as fh:
            digests[rel] = hashlib.sha256(fh.read()).hexdigest()
    with open(os.path.join(HERE, 'reference_checkout_sha256.json'), 'w') as fh:
        json.dump(digests, fh, indent=1, sort_keys=True)
        fh.write('\n')
    print('reference test fixtures refreshed under', dst)


def spread_lambda_fixture():
    """spreadLambdaProtocol (blues/utils.py:276-369) for the schedules and step counts tests/test_host_logic.py checks →
    spread_lambda_protocol.json.  With BLUES_REFERENCE_DATA set the reference's function runs from its source text;
    without it, this package's utils.spreadLambdaProtocol does, and ``source`` records which."""
    import ast
    import json
    from scipy.interpolate import interp1d
    from tests.test_host_logic import SPREAD_LAMBDA_CASES
    if REF:
        path = os.path.join(os.path.dirname(os.path.dirname(REF)), 'utils.py')
        tree = ast.parse(open(path).read())
        fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == 'spreadLambdaProtocol'][0]
        ns = {'np': np, 'interp1d': interp1d, 'floor': math.floor}
        exec(compile(ast.Module([fn], []), path, 'exec'), ns)
        spread, source = ns['spreadLambdaProtocol'], 'reference blues/utils.py spreadLambdaProtocol'
    else:
        from blues_b200 import utils
        spread, source = utils.spreadLambdaProtocol, 'blues_b200.utils.spreadLambdaProtocol'
    out = {'source': source, 'tables': {}}
    for name, vals, kind, n in SPREAD_LAMBDA_CASES:
        out['tables']['%s/%s/%d' % (name, kind, n)] = [float(v) for v in spread(list(vals), n, switching_types=kind,
                                                                                 return_tab_function=False)]
    with open(os.path.join(HERE, 'spread_lambda_protocol.json'), 'w') as f:
        json.dump(out, f)
        f.write('\n')
    print('spreadLambdaProtocol tables:', len(out['tables']), 'from', source)


def main():
    if '--spread-lambda' in sys.argv:
        return spread_lambda_fixture()
    if not REF:
        raise SystemExit('set BLUES_REFERENCE_DATA to <MobleyLab/blues checkout>/blues/tests/data')
    if '--reference-tests' in sys.argv:
        return reference_tests()
    reference_bookkeeping()
    ethylene_fixture()
    structs = {}
    for out, base in (('tol_parm', 'TOL-parm'), ('wat_divaline', 'watDivaline'), ('vac_divaline', 'vacDivaline')):
        s = load_file(os.path.join(REF, base + '.prmtop'), xyz=os.path.join(REF, base + '.inpcrd'))
        s.save_npz(os.path.join(HERE, out + '.npz'))
        structs[out] = s
        print(out, s.n_atoms)
    t4l = build_t4l_surrogate()
    t4l.save_npz(os.path.join(HERE, 't4l_surrogate.npz'))
    print('t4l_surrogate', t4l.n_atoms, 'bonds', len(t4l.bonds), 'angles', len(t4l.angles), 'dihedrals', len(t4l.dihedrals),
          'net charge %.6f' % t4l.charges.sum())
    if '--no-vectors' not in sys.argv:
        vec = oracle_vectors(structs)
        np.savez_compressed(os.path.join(HERE, 'oracle_vectors.npz'), **vec)
        print('oracle vectors:', len(vec))


if __name__ == '__main__':
    main()
