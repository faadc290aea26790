#!/usr/bin/env python
"""Fixture for tests/test_openmm_adapter.py: the COMPLETE forces that the reference's AbsoluteAlchemicalFactory builds for
the three configurations of make_alchemy_golden.py (every particle parameter, interaction group, global parameter, flag),
serialised so that machines without the reference's source can rebuild the stand-in objects and feed them to
contrib.openmm_adapter.  Needs the reference's source (make_alchemy_golden.load_factory).  Output:
tests/golden/adapter_forces.json, and the SHA-256 of each configuration's forces as the reference factory built them in
tests/golden/adapter_forces_sha256.json (what the test compares the fixture with)."""
import hashlib, json, os, sys
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE); sys.path.insert(0, os.path.join(HERE, '..')); sys.path.insert(0, os.path.join(HERE, '..', '..'))
import make_alchemy_golden as g
from openmmtools_b200 import unit as u
from helpers import lj_setup


GPU_RC, GPU_RS = 0.75, 0.68   # nm; L = 1.578 nm for 40 particles at reduced density 0.4


def dump(f):
    d = {'type': type(f).__name__, 'globals': dict(f.globals)}
    if isinstance(f, g.NonbondedForce):
        d.update(particles=[[float(u.to_md(x)) for x in p] for p in f.particles], exceptions=len(f.exceptions), method=f.method,
                 cutoff=float(u.to_md(f.cutoff)), use_switch=bool(f.use_switch), switch_distance=float(u.to_md(f.switch_distance)),
                 dispersion=bool(f.dispersion))
    elif isinstance(f, g.CustomNonbondedForce):
        d.update(expression=f.expression, per_particle=f.per_particle, particles=[[float(u.to_md(x)) for x in p] for p in f.particles],
                 groups=[[list(a), list(b)] for a, b in f.groups], method=f.method, cutoff=float(u.to_md(f.cutoff)),
                 use_switch=bool(f.use_switch), switch_distance=float(u.to_md(f.switch_distance)), lrc=bool(f.lrc))
    else:
        d.update(expression=f.expression, n_bonds=len(f.bonds))
    return d


def digest(forces):
    """SHA-256 of one configuration's dumped forces in canonical JSON."""
    return hashlib.sha256(json.dumps(forces, sort_keys=True).encode()).hexdigest()


if __name__ == '__main__':
    Factory, Region = g.load_factory()
    s = lj_setup(N=g.N, n_alch=g.N_ALCH, reduced_density=0.4, seed=77)
    out, sha = {}, {}
    for c, (annihilate, disable_lrc, (alpha, a, b, cc)) in enumerate(g.CONFIGS):
        factory = Factory(disable_alchemical_dispersion_correction=disable_lrc)
        region = Region(alchemical_atoms=list(range(g.N_ALCH)), annihilate_sterics=annihilate, softcore_alpha=alpha,
                        softcore_a=a, softcore_b=b, softcore_c=cc)
        forces = factory._alchemically_modify_NonbondedForce(g.reference_force(s), [region], frozenset())
        out['config%d' % c] = [dump(f) for v in forces.values() for f in v]
        sha['config%d' % c] = digest(json.loads(json.dumps(out['config%d' % c])))
        # The same forces with a cutoff the engine (like OpenMM) accepts in this small box (r_c <= L/2): the energies the
        # GPU test compares with, again evaluated from the reference-emitted expressions inside the cutoff.
        U = []
        for lam in g.LAMBDAS:
            e = 0.0
            for v in forces.values():
                for f in v:
                    f.cutoff = GPU_RC * u.nanometer
                    if isinstance(f, g.NonbondedForce):
                        e += g.nonbonded_energy(f, s['x'], s['L'])
                    elif isinstance(f, g.CustomNonbondedForce):
                        e += g.custom_nonbonded_energy(f, s['x'], s['L'], {'lambda_sterics': lam, 'lambda_electrostatics': lam})
            U.append(e)
        out['config%d_U_gpu' % c] = U
    out['gpu_rc'] = GPU_RC
    out['gpu_rs'] = GPU_RS
    dst = os.path.join(HERE, 'adapter_forces.json')
    json.dump(out, open(dst, 'w'))
    print('wrote', dst, os.path.getsize(dst))
    dst = os.path.join(HERE, 'adapter_forces_sha256.json')
    json.dump(sha, open(dst, 'w'), indent=1)
    print('wrote', dst)
