"""A/B timing of the swap-all walker builds on one GPU (development aid).
  python tools/ab_walk.py libA.so libB.so ...     each library runs in its own process (RX_B200_LIB), K = 256 on the
  real alchemical-LJ energy matrix tools/data/u_lj_256.npy; prints walker ms, rounds, ns/round and a permutation digest
  (all builds must print the same digest)."""
import os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r'''
import sys, os, zlib
sys.path.insert(0, %r)
import numpy as np
from openmmtools_b200._engine import Engine
K = int(os.environ.get('AB_K', '256'))
u = np.load(os.path.join(%r, 'tools', 'data', 'u_lj_256.npy'))[:K, :K].copy()
e = Engine(0, K, K, 0)
e.set_energies(u); e.set_replica_states(np.arange(K)); e.mix_seed(1234, 0)
out = []
for rep in range(int(os.environ.get('AB_REPS', '3'))):
    st, nacc, nprop = e.mix_swap_all(K ** 3)
    ms = e.mix_stats()
    out.append((ms['walker_ms'], ms['rounds'], zlib.crc32(st.tobytes()) ^ zlib.crc32(nacc.tobytes()) ^ zlib.crc32(nprop.tobytes())))
best = min(o[0] for o in out)
print('walker %%8.2f ms (best of %%d)  rounds %%d  %%6.1f ns/round  digests %%s' %% (best, len(out), out[-1][1], 1e6 * best / max(out[-1][1], 1), ' '.join('%%08x' %% o[2] for o in out)))
''' % (ROOT, ROOT)

for lib in sys.argv[1:]:
    env = dict(os.environ)
    if lib != 'default':
        env['RX_B200_LIB'] = os.path.abspath(lib)
    try:
        r = subprocess.run([sys.executable, '-c', CHILD], env=env, capture_output=True, text=True, timeout=int(os.environ.get('AB_TIMEOUT', '90')))
        print('%-28s %s' % (os.path.basename(lib), (r.stdout.strip() or r.stderr.strip()[-400:])))
    except subprocess.TimeoutExpired:
        print('%-28s TIMEOUT' % os.path.basename(lib))
    sys.stdout.flush()
