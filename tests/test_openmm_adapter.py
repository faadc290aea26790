"""contrib.openmm_adapter: the forces the REFERENCE's AbsoluteAlchemicalFactory builds (class body lifted from the
reference's alchemy/alchemy.py by tests/golden/make_alchemy_golden.py, run on recording OpenMM stand-ins, stored in
tests/golden/adapter_forces.json) are read back into the engine's parameter record; on the GPU the engine built
from that record reproduces the golden energies of tests/golden/alchemy_golden.npz (evaluated with numpy from the
reference-emitted expressions)."""
import json
import os
import sys
import numpy as np
import pytest
from openmmtools_b200 import unit as u
from openmmtools_b200.contrib import openmm_adapter as adapter
from helpers import lj_setup, KB

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, 'golden'))
G = np.load(os.path.join(HERE, 'golden', 'alchemy_golden.npz'))


class StandInSystem:
    """What system_from_openmm reads besides the forces."""

    def __init__(self, s):
        self.s = s

    def getParticleMass(self, i):
        return self.s['mass'][i] * u.dalton

    def getDefaultPeriodicBoxVectors(self):
        L = self.s['L']
        return [np.array(v) * u.nanometer for v in ([L, 0, 0], [0, L, 0], [0, 0, L])]


CONFIGS = [(False, False, (0.5, 1, 1, 6)), (True, False, (0.5, 1, 1, 6)), (False, True, (0.3, 2, 1.5, 12))]   # make_alchemy_golden.py
N, N_ALCH, LAMBDAS = 40, 6, [0.0, 0.3, 0.7, 1.0]
FIXTURE = json.load(open(os.path.join(HERE, 'golden', 'adapter_forces.json')))
LIFT_SHA256 = json.load(open(os.path.join(HERE, 'golden', 'adapter_forces_sha256.json')))


class _Stub:
    """A force rebuilt from the fixture, with the OpenMM getters the adapter uses."""
    CutoffPeriodic = 2

    def __init__(self, d):
        self.d = d
        self.globals = d['globals']
        self.expression = d.get('expression')
        self.particles = d.get('particles', [])
        self.groups = [(a, b) for a, b in d.get('groups', [])]
        self.lrc = d.get('lrc')
        self.bonds = [None] * d.get('n_bonds', 0)

    def getNumParticles(self): return len(self.particles)
    def getParticleParameters(self, i): return list(self.particles[i])
    def getNumExceptions(self): return self.d['exceptions']
    def getNonbondedMethod(self): return self.d['method']
    def getCutoffDistance(self): return self.d['cutoff']
    def getUseSwitchingFunction(self): return self.d['use_switch']
    def getSwitchingDistance(self): return self.d['switch_distance']
    def getUseDispersionCorrection(self): return self.d['dispersion']


def fixture_forces(c, cutoff=None, switch=None):
    out = []
    for d in json.loads(json.dumps(FIXTURE['config%d' % c])):   # a private copy: a test may edit it
        if cutoff is not None and 'cutoff' in d:
            d['cutoff'], d['switch_distance'] = cutoff, switch
        f = type(d['type'], (_Stub,), {})(d)     # the adapter dispatches on the class NAME
        out.append(f)
    return lj_setup(N=N, n_alch=N_ALCH, reduced_density=0.4, seed=77), out


def test_fixture_equals_a_fresh_lift_of_the_reference_factory():
    """Every configuration of the fixture is, to the last digit, what the lifted reference factory built: the SHA-256 of
    each configuration's forces was recorded from that lift (tests/golden/make_adapter_golden.py)."""
    import make_alchemy_golden as g
    import make_adapter_golden as m
    assert g.CONFIGS == CONFIGS and (g.N, g.N_ALCH, g.LAMBDAS) == (N, N_ALCH, LAMBDAS)
    assert sorted(LIFT_SHA256) == ['config%d' % c for c in range(len(CONFIGS))]
    for c in range(len(CONFIGS)):
        assert m.digest(FIXTURE['config%d' % c]) == LIFT_SHA256['config%d' % c], c


@pytest.mark.parametrize('c', [0, 1, 2])
def test_record_from_reference_factory_forces(c):
    s, forces = fixture_forces(c)
    annihilate, disable_lrc, soft = CONFIGS[c]
    rec = adapter.system_from_openmm(StandInSystem(s), forces)
    assert rec.alchemical_atoms == tuple(range(N_ALCH))
    assert rec.annihilate_sterics == annihilate
    assert (rec.softcore_alpha, rec.softcore_a, rec.softcore_b, rec.softcore_c) == tuple(float(x) for x in soft)
    assert rec.alchemical_dispersion_correction == (not disable_lrc)
    assert np.allclose(rec.sigma, s['sigma']) and np.allclose(rec.epsilon, s['eps'])      # alchemical epsilons restored
    assert rec.cutoff == pytest.approx(s['rc']) and not rec.use_switching_function
    assert np.allclose(rec.box_vectors, np.eye(3) * s['L'])
    # the same record as our own factory builds from our own LJ record
    desc = json.loads(str(G['config%d_forces' % c]))
    assert any(f['type'] == 'CustomNonbondedForce' for v in desc.values() for f in v)


def test_plain_lj_force_and_refusals():
    s, forces = fixture_forces(0)
    nb = [f for f in forces if type(f).__name__ == 'NonbondedForce']
    rec = adapter.system_from_openmm(StandInSystem(s), nb)
    assert not rec.is_alchemical and rec.epsilon[0] == 0.0        # without the custom forces the zeroed epsilons stay
    nb[0].particles[3][0] = 0.5
    with pytest.raises(NotImplementedError):
        adapter.system_from_openmm(StandInSystem(s), nb)


@pytest.mark.gpu
@pytest.mark.parametrize('c', [0, 1, 2])
def test_engine_from_adapter_reproduces_reference_energies(c):
    # (the factory's forces with a cutoff the engine -- like OpenMM -- accepts in this small box: r_c <= L/2)
    s, forces = fixture_forces(c, FIXTURE['gpu_rc'], FIXTURE['gpu_rs'])
    rec = adapter.system_from_openmm(StandInSystem(s), forces)
    assert rec.cutoff == FIXTURE["gpu_rc"]
    # the golden numbers are the reference-emitted expressions inside the cutoff: no long-range corrections
    rec.use_dispersion_correction = False
    rec.alchemical_dispersion_correction = False
    from openmmtools_b200 import _backend
    tstates = adapter.thermodynamic_states_from_openmm(rec, [300.0] * len(LAMBDAS), LAMBDAS)
    eng = _backend.build_engine(tstates, 1)
    eng.set_positions(G['x'][None])
    u_row = eng.compute_energies()[0] * (KB * 300.0)
    eng.close()
    ref = np.array(FIXTURE['config%d_U_gpu' % c])
    assert np.abs(u_row - ref).max() <= 1e-9 * max(1.0, np.abs(ref).max()), (u_row, ref)
