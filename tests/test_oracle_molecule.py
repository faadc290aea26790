"""The small-molecule path on the CPU: the AMBER reader and the fixture of testsystems.AlanineDipeptideVacuum
(testsystems.py:3352-3388), the oracle's force field (forces = -grad U by finite differences) and its constrained Langevin
steps (integrators.py:1404-1460).  Parity with OpenMM itself is unpinned (not installable here); the energy at the input
geometry is pinned to this implementation's own value so that a regression shows."""
import copy
import json
import os
import sys
import numpy as np
from openmmtools_b200 import testsystems, unit, amber
from oracle import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
KB = 8.31446261815324e-3


def aladip():
    a = testsystems.AlanineDipeptideVacuum()
    return a, np.ascontiguousarray(a.positions.value_in_unit(unit.nanometer), np.float64)


def test_fixture_equals_a_fresh_parse_of_the_reference_files():
    """The packaged parameters are what the AMBER reader makes of the original project's prmtop/crd (tests/golden)."""
    sys.path.insert(0, os.path.join(HERE, 'golden'))
    import make_aladip_fixture as m
    fresh = json.loads(json.dumps(m.build()))
    stored = json.load(open(os.path.join(HERE, '..', 'openmmtools_b200', 'data', 'alanine_dipeptide_vacuum.json')))
    assert fresh == stored


def test_topology_counts_and_units():
    a, x = aladip()
    s = a.system
    assert s.n_particles == 22 and a.atom_names[:4] == ['HH31', 'CH3', 'HH32', 'HH33']
    assert abs(s.charge.sum()) < 1e-8 and abs(s.masses.sum() - 144.176) < 1e-9
    assert len(s.constraints) == 12 and len(s.bonds) == 9 and len(s.angles) == 36 and len(s.torsions) == 32
    assert len(s.exclusions) == 57 and len(s.exceptions) == 41 and s.getNumConstraints() == 12
    # every constrained bond involves a hydrogen and has its AMBER length; the input geometry satisfies it to 1e-7 nm
    for i, j, d in s.constraints:
        assert min(s.masses[int(i)], s.masses[int(j)]) < 1.1
        assert abs(np.linalg.norm(x[int(i)] - x[int(j)]) - d) < 2e-7
    # ff96 numbers: CT sigma 3.39967 A, epsilon 0.1094 kcal/mol; C-N bond 490 kcal/mol/A^2 at 1.335 A
    assert abs(s.sigma[1] - 0.339967) < 1e-6 and abs(s.epsilon[1] - 0.1094 * 4.184) < 1e-6
    cn = [b for b in s.bonds if {int(b[0]), int(b[1])} == {4, 6}][0]
    assert abs(cn[2] - 2 * 490.0 * 418.4) < 1e-6 and abs(cn[3] - 0.1335) < 1e-12
    # 1-4 pairs: Coulomb / 1.2, Lennard-Jones epsilon / 2
    i, j, qq, sg, ep = s.exceptions[0]
    i, j = int(i), int(j)
    assert abs(qq - s.charge[i] * s.charge[j] / 1.2) < 1e-15
    assert abs(ep - np.sqrt(s.epsilon[i] * s.epsilon[j]) / 2.0) < 1e-9 and abs(sg - 0.5 * (s.sigma[i] + s.sigma[j])) < 1e-9
    none = testsystems.AlanineDipeptideVacuum(constraints=None).system
    assert len(none.constraints) == 0 and len(none.bonds) == 21


def test_oracle_forces_are_the_gradient_of_the_energy():
    a, x = aladip()
    x = x + np.random.default_rng(0).normal(0, 0.005, x.shape)
    for constraints in ('HBonds', None):
        m = oracle.Molecule(testsystems.AlanineDipeptideVacuum(constraints=constraints).system)
        U, f = m.energy(x, forces=True)
        g = np.zeros_like(x); h = 1e-6
        for i in range(22):
            for c in range(3):
                xp = x.copy(); xp[i, c] += h; xm = x.copy(); xm[i, c] -= h
                g[i, c] = -(m.energy(xp) - m.energy(xm)) / (2 * h)
        assert np.abs(g - f).max() < 1e-5 * np.abs(f).max()
        assert np.abs(f.sum(0)).max() < 1e-8      # no net force


def test_energy_at_the_input_geometry_is_pinned():
    a, x = aladip()
    U = oracle.Molecule(a.system).energy(x)
    assert abs(U - (-88.08858703851178)) < 1e-9      # kJ/mol (this implementation's own value: -21.0537 kcal/mol)
    # each term alone (kcal/mol): bonds without H, angles, torsions, nonbonded incl. 1-4
    s0 = a.system
    parts = {}
    for name in ('bonds', 'angles', 'torsions'):
        s = copy.deepcopy(s0)
        for other in ('bonds', 'angles', 'torsions'):
            if other != name: setattr(s, other, np.zeros((0, getattr(s, other).shape[1])))
        s.charge = np.zeros(22); s.epsilon = np.zeros(22); s.exceptions = np.zeros((0, 5))
        parts[name] = oracle.Molecule(s).energy(x) / 4.184
    assert 0.0 <= parts['bonds'] < 0.1 and 0.2 < parts['angles'] < 0.6 and 1.0 < parts['torsions'] < 12.0


def test_constrained_langevin_keeps_the_constraints_and_the_temperature():
    a, x = aladip()
    m = oracle.Molecule(a.system)
    kT = KB * 300.0
    rng = np.random.default_rng(1)
    v = np.ascontiguousarray(rng.normal(size=x.shape) * np.sqrt(kT / m.mass)[:, None])
    n = 4000
    kes = []
    for block in range(8):
        m.langevin(x, v, rng.normal(size=(n // 8, 22, 3)), kT, 0.002, 5.0, n // 8, 'VRORV', tol=1e-10)
        kes.append(m.kinetic(v))
    c = a.system.constraints
    i, j = c[:, 0].astype(int), c[:, 1].astype(int)
    assert np.abs(np.linalg.norm(x[i] - x[j], axis=1) - c[:, 2]).max() < 1e-10
    assert np.abs(((x[i] - x[j]) * (v[i] - v[j])).sum(1)).max() < 1e-9
    # 66 - 12 constraints - 3 (centre of mass) degrees of freedom
    assert abs(np.mean(kes) / (0.5 * kT * 51) - 1.0) < 0.5
    assert np.isfinite(m.energy(x))
