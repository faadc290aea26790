"""One swap-all call (for ncu captures of the walkers): the K=256 LJ energy matrix, or with K given, a K x K matrix sampled
from its rows and columns (rows repeat above K = 256); K not a power of two runs k_mix_walk2c below 256 and k_mix_walk_any
above.  usage: mix_once.py [nswap [K]]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from openmmtools_b200._engine import Engine
K = int(sys.argv[2]) if len(sys.argv) > 2 else 256
u = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'data', 'u_lj_256.npy'))
if K != 256:
    idx = np.linspace(0, 255, K).round().astype(int)
    u = np.ascontiguousarray(u[np.ix_(idx, idx)])
e = Engine(0, K, K, 0)
e.set_energies(u); e.set_replica_states(np.arange(K)); e.mix_seed(1234, 0)
n = int(sys.argv[1]) if len(sys.argv) > 1 else K ** 3 // 8
e.mix_swap_all(n)
print(e.mix_stats())
