"""k_propagate (float32 state, one CTA per replica) against the double-precision oracle integrator fed with the
same Philox noise.  Dynamics cannot be compared with OpenMM bit for bit (its Gaussian stream is internal), so
parity is: identical update rule on identical inputs and noise, to float32 accuracy."""
import numpy as np
import pytest
from helpers import lj_setup, oracle_system, gpu_engine, KB, device_noise, device_reassign_noise

pytestmark = pytest.mark.gpu


def make_engine(s, K, M, lambdas, temps, dt, gamma, n_steps, splitting):
    e = gpu_engine(1, K, M, s['N'], box=(s['L'],) * 3, r_cutoff=s['rc'], r_switch=s['rs'], use_switch=True)
    e.set_particles(s['sigma'], s['eps'], s['mass'], s['alch'])
    e.set_states(temps, lambdas)
    e.set_integrator(dt, gamma, n_steps, splitting)
    return e


@pytest.mark.parametrize('splitting,n_steps', [('V R O R V', 1), ('V R O R V', 8), ('O V R V O', 4), ('R V O', 3),
                                               ('V R R O R R V', 2)])
def test_steps_match_oracle_with_same_noise(splitting, n_steps):
    N, K, M = 256, 4, 4
    s = lj_setup(N=N, n_alch=6, seed=11)
    lambdas = np.array([1.0, 0.6, 0.3, 0.0]); temps = np.array([300.0, 310.0, 320.0, 330.0])
    dt, gamma = 0.002, 10.0
    e = make_engine(s, K, M, lambdas, temps, dt, gamma, n_steps, splitting)
    rng = np.random.default_rng(2)
    x0 = np.stack([s['x']] * K)
    v0 = rng.normal(scale=0.25, size=(K, N, 3)).astype(np.float32).astype(np.float64)
    e.set_positions(x0); e.set_velocities(v0)
    states = np.array([2, 0, 3, 1])
    e.set_replica_states(states)
    seed, iteration = 0x1234567890ABCDEF, 7
    e.propagate(seed, iteration)
    xg = e.get_positions(); vg = e.get_velocities()
    pot, kin = e.get_replica_energies()
    osys = oracle_system(s)
    prog = splitting.replace(' ', '')
    nO = prog.count('O')
    for k in range(K):
        x = x0[k].copy(); v = v0[k].copy()
        noise = device_noise(seed, iteration, k, N, n_steps * nO)
        U = osys.langevin(x, v, noise, lambdas[states[k]], KB * temps[states[k]], dt, gamma, n_steps, prog)
        xw = x - s['L'] * np.floor(x / s['L'])
        d = xg[k] - xw
        d -= s['L'] * np.round(d / s['L'])
        assert np.abs(d).max() < 2e-5, (k, np.abs(d).max())
        assert np.abs(vg[k] - v).max() < 2e-4, (k, np.abs(vg[k] - v).max())
        assert abs(pot[k] - U) < 1e-3 * max(1.0, abs(U)), (pot[k], U)
        ke = 0.5 * (s['mass'][:, None] * v * v).sum()
        assert abs(kin[k] - ke) < 1e-4 * ke
    e.close()


def test_reassign_velocities_uses_maxwell_boltzmann():
    N, K, M = 512, 8, 8
    s = lj_setup(N=N, n_alch=10, seed=12)
    temps = np.linspace(250, 400, M); lambdas = np.ones(M)
    e = make_engine(s, K, M, lambdas, temps, 0.001, 10.0, 0, 'V R O R V')
    e.set_positions(np.stack([s['x']] * K))
    e.set_replica_states(np.arange(K))
    e.propagate(99, 3, reassign_velocities=True)
    v = e.get_velocities()
    for k in range(K):
        g = device_reassign_noise(99, 3, k, N)
        ref = np.sqrt(KB * temps[k] / s['mass'][0]) * g
        assert np.abs(v[k] - ref).max() < 1e-5
        T_kin = (s['mass'][:, None] * v[k] ** 2).sum() / (3 * N * KB)
        assert abs(T_kin / temps[k] - 1) < 0.15
    e.close()


def test_harmonic_oscillator_steps():
    from oracle import oracle
    N, K, M = 1, 3, 3
    e = gpu_engine(2, K, M, N)
    mass = np.array([39.948])
    e.set_particles(None, None, mass, None)
    Ks = np.array([100.0, 200.0, 400.0]) * 4.184 * 100
    x0s = np.array([[0.0, 0, 0], [0.1, 0, 0], [0.0, -0.1, 0.05]])
    temps = np.array([300.0, 310.0, 320.0])
    e.set_states(temps, None, np.array([0.0, 1.0, 2.0]), Ks, x0s)
    n_steps, dt, gamma = 50, 0.001, 10.0
    e.set_integrator(dt, gamma, n_steps, 'V R O R V')
    x0 = np.array([[[0.01, 0.02, -0.01]], [[0.1, 0.0, 0.0]], [[0.0, 0.0, 0.0]]])
    v0 = np.array([[[0.1, -0.2, 0.3]], [[0.0, 0.1, 0.0]], [[0.2, 0.2, 0.2]]])
    e.set_positions(x0); e.set_velocities(v0)
    e.set_replica_states(np.array([1, 2, 0]))
    e.propagate(5, 0)
    xg, vg = e.get_positions(), e.get_velocities()
    pot, kin = e.get_replica_energies()
    st = [1, 2, 0]
    for k in range(K):
        x = x0[k].astype(np.float32).astype(np.float64); v = v0[k].astype(np.float32).astype(np.float64)
        noise = device_noise(5, 0, k, N, n_steps)
        U = oracle.ho_langevin(x, v, mass, noise, Ks[st[k]], x0s[st[k]], [0.0, 1.0, 2.0][st[k]], KB * temps[st[k]], dt,
                               gamma, n_steps)
        assert np.abs(xg[k] - x).max() < 1e-5
        assert np.abs(vg[k] - v).max() < 1e-4
        assert abs(pot[k] - U) < 1e-4 * max(1, abs(U))
    # energies: u[k,l] = beta_l (K_l/2 |x-x0_l|^2 + U0_l)
    u = e.compute_energies()
    for k in range(K):
        for l in range(M):
            ref = (0.5 * Ks[l] * ((xg[k][0] - x0s[l]) ** 2).sum() + [0.0, 1.0, 2.0][l]) / (KB * temps[l])
            assert abs(u[k, l] - ref) < 1e-5 * max(1, abs(ref))
    e.close()


def test_neighbour_list_run_equals_all_pairs_run(monkeypatch):
    """300 hot 2-fs steps (the inner list is re-partitioned many times, the outer list rebuilt, atoms re-dealt to
    threads) against the same launch with the all-pairs force loop: a pair missing from a list would show up as a
    different trajectory; only the float32 summation order differs between the two."""
    N, K, M = 256, 3, 3
    s = lj_setup(N=N, n_alch=6, seed=21)
    lambdas = np.array([1.0, 0.5, 0.0]); temps = np.array([600.0, 600.0, 600.0])
    rng = np.random.default_rng(5)
    v0 = rng.normal(scale=0.35, size=(K, N, 3)).astype(np.float32).astype(np.float64)
    out = []
    for no_list in (False, True):
        if no_list:
            monkeypatch.setenv('RX_NO_VERLET', '1')
        e = make_engine(s, K, M, lambdas, temps, 0.002, 1.0, 300, 'V R O R V')
        e.set_positions(np.stack([s['x']] * K)); e.set_velocities(v0)
        e.set_replica_states(np.arange(K))
        e.propagate(99, 3)
        out.append((e.get_positions(), e.get_velocities(), e.get_replica_energies()[0]))
        e.close()
    (xa, va, pa), (xb, vb, pb) = out
    d = xa - xb
    d -= s['L'] * np.round(d / s['L'])
    assert np.abs(d).max() < 2e-3, np.abs(d).max()           # chaotic growth of float32 round-off, not a missed pair
    assert np.median(np.abs(d)) < 2e-5
    assert np.abs(pa - pb).max() < 0.05 * max(1.0, np.abs(pb).max())


def test_dense_fluid_falls_back_to_all_pairs_and_matches_oracle():
    """Liquid density: more neighbours than a list column holds -> the CTA switches to the all-pairs loop."""
    N, K, M = 256, 2, 2
    s = lj_setup(N=N, n_alch=4, reduced_density=0.6, seed=31)
    lambdas = np.array([1.0, 0.4]); temps = np.array([300.0, 300.0])
    dt, gamma, n_steps = 0.001, 10.0, 4
    e = make_engine(s, K, M, lambdas, temps, dt, gamma, n_steps, 'V R O R V')
    x0 = np.stack([s['x']] * K)
    v0 = np.random.default_rng(8).normal(scale=0.2, size=(K, N, 3)).astype(np.float32).astype(np.float64)
    e.set_positions(x0); e.set_velocities(v0); e.set_replica_states(np.arange(K))
    e.propagate(5, 1)
    xg, vg = e.get_positions(), e.get_velocities()
    osys = oracle_system(s)
    for k in range(K):
        x = x0[k].copy(); v = v0[k].copy()
        osys.langevin(x, v, device_noise(5, 1, k, N, n_steps), lambdas[k], KB * temps[k], dt, gamma, n_steps, 'VRORV')
        d = xg[k] - (x - s['L'] * np.floor(x / s['L']))
        d -= s['L'] * np.round(d / s['L'])
        assert np.abs(d).max() < 5e-5, (k, np.abs(d).max())
        # forces of a dense, roughly packed start are large: velocities to float32 accuracy of those forces
        assert np.abs(vg[k] - v).max() < 1e-3 * max(1.0, np.abs(v).max()), (k, np.abs(vg[k] - v).max())
    e.close()


@pytest.mark.parametrize('use_switch,annihilate,alpha,a,b,c', [(False, False, 0.5, 1.0, 1.0, 6.0), (True, True, 0.5, 1.0, 1.0, 6.0),
                                                                (True, False, 0.3, 2.0, 1.5, 12.0), (False, True, 0.7, 1.0, 2.0, 4.0)])
def test_pair_kernel_variants_match_oracle(use_switch, annihilate, alpha, a, b, c):
    """Every specialisation of the pair function (switch on/off, softcore_c == 6 or not) and the annihilating A-A
    pairs, 6 steps against the oracle with the same noise (alchemy.py:1383-1388 energy expression)."""
    N, K, M = 256, 3, 3
    s = lj_setup(N=N, n_alch=8, seed=41)
    lambdas = np.array([0.8, 0.45, 0.1]); temps = np.array([300.0, 300.0, 300.0])
    dt, gamma, n_steps = 0.002, 5.0, 6
    e = gpu_engine(1, K, M, N, box=(s['L'],) * 3, r_cutoff=s['rc'], r_switch=s['rs'], use_switch=use_switch,
                   annihilate_sterics=annihilate, softcore_alpha=alpha, softcore_a=a, softcore_b=b, softcore_c=c)
    e.set_particles(s['sigma'], s['eps'], s['mass'], s['alch'])
    e.set_states(temps, lambdas)
    e.set_integrator(dt, gamma, n_steps, 'V R O R V')
    x0 = np.stack([s['x']] * K)
    v0 = np.random.default_rng(3).normal(scale=0.25, size=(K, N, 3)).astype(np.float32).astype(np.float64)
    e.set_positions(x0); e.set_velocities(v0); e.set_replica_states(np.arange(K))
    e.propagate(11, 2)
    xg, vg = e.get_positions(), e.get_velocities()
    pot = e.get_replica_energies()[0]
    osys = oracle_system(s, annihilate=annihilate, alpha=alpha, a=a, b=b, c=c, use_switch=use_switch)
    for k in range(K):
        x = x0[k].copy(); v = v0[k].copy()
        U = osys.langevin(x, v, device_noise(11, 2, k, N, n_steps), lambdas[k], KB * temps[k], dt, gamma, n_steps, 'VRORV')
        d = xg[k] - (x - s['L'] * np.floor(x / s['L']))
        d -= s['L'] * np.round(d / s['L'])
        assert np.abs(d).max() < 2e-5, (k, np.abs(d).max())
        assert np.abs(vg[k] - v).max() < 3e-4, (k, np.abs(vg[k] - v).max())
        assert abs(pot[k] - U) < 2e-3 * max(1.0, abs(U)), (pot[k], U)
    e.close()


def test_cluster_split_replica_reproduces_single_block_trajectory():
    """A replica split over a thread-block cluster (atoms partitioned over 4 blocks, positions exchanged through
    distributed shared memory, cluster-wide displacement votes) must give the SAME trajectory as one block per replica:
    lists are rebuilt at the same steps with the same contents, every atom sums its own list in list order, noise is
    keyed by atom id.  Engine A (3 replicas) runs in clusters of four; engine B has too many replicas for that and runs
    one block per replica, its first 3 replicas starting where A's do.  200 hot steps cross several re-partitions and
    at least one outer rebuild."""
    import torch
    N, K = 512, 3
    s = lj_setup(N=N, n_alch=10, seed=51)
    lambdas = np.array([1.0, 0.5, 0.0]); temps = np.array([500.0, 500.0, 500.0])
    rng = np.random.default_rng(15)
    n_b = torch.cuda.get_device_properties(0).multi_processor_count // 4 + 1
    v0 = rng.normal(scale=0.3, size=(n_b, N, 3)).astype(np.float32).astype(np.float64)
    out = []
    for n in (K, n_b):
        e = make_engine(s, n, K, lambdas, temps, 0.002, 1.0, 200, 'V R O R V')
        e.set_positions(np.stack([s['x']] * n)); e.set_velocities(v0[:n])
        e.set_replica_states(np.array([1, 2, 0] + [k % K for k in range(K, n)]))
        e.propagate(1234, 9)
        x, v, (pe, ke) = e.get_positions(), e.get_velocities(), e.get_replica_energies()
        out.append((x[:K], v[:K], (pe[:K], ke[:K])))
        e.close()
    (xa, va, (pa, ka)), (xb, vb, (pb, kb)) = out
    assert np.array_equal(xa, xb) and np.array_equal(va, vb)
    assert np.allclose(pa, pb, rtol=1e-12, atol=1e-9) and np.allclose(ka, kb, rtol=1e-12, atol=1e-9)   # other summation order


@pytest.mark.parametrize('splitting,code', [('', 'INVALID'), ('VR', 'INVALID'), ('VRXO', 'UNSUPPORTED'),
                                             ('VRO' * 10 + 'VR', 'INVALID')])
def test_bad_splitting_is_refused_alike_for_one_move_and_per_state_moves(splitting, code):
    """rx_set_integrator and rx_set_state_integrator check a splitting with the same rules: empty, without O, with an
    unknown substep, 32 substeps."""
    from openmmtools_b200 import _lib
    from openmmtools_b200._engine import EngineError
    e = gpu_engine(2, 2, 2, 1)
    e.set_integrator(0.001, 1.0, 10, 'V R O R V')
    with pytest.raises(EngineError) as one:
        e.set_integrator(0.001, 1.0, 10, splitting)
    with pytest.raises(EngineError) as per_state:
        e.set_state_integrator(0, 0.001, 1.0, 10, splitting)
    assert one.value.code == per_state.value.code == getattr(_lib, 'RX_ERR_' + code)
    assert one.value.message.startswith('rx_set_integrator:')
    assert per_state.value.message.startswith('rx_set_state_integrator:')
    e.close()


def test_per_state_moves_propagate_each_replica_with_the_move_of_its_state():
    """One MCMCMove per thermodynamic state (multistatesampler.py:906-910, :1311-1322): in ONE launch the replicas in states
    0, 1 run move A and those in states 2, 3 move B (other timestep, friction, step count, splitting, velocity
    reassignment).  Each replica must come out exactly as from an engine where every state has that move."""
    N, K = 256, 4
    s = lj_setup(N=N, n_alch=8, seed=61)
    lambdas = np.array([1.0, 0.7, 0.3, 0.0]); temps = np.array([300.0, 320.0, 340.0, 360.0])
    A = (0.002, 1.0, 40, 'V R O R V', False)
    B = (0.001, 5.0, 25, 'O V R V O', True)
    rng = np.random.default_rng(16)
    v0 = rng.normal(scale=0.3, size=(K, N, 3)).astype(np.float32).astype(np.float64)
    perm = np.array([2, 0, 3, 1])            # replica -> state
    def run(moves):
        e = make_engine(s, K, K, lambdas, temps, *moves[0][:4])
        if any(m != moves[0] for m in moves):
            for l, m in enumerate(moves):
                e.set_state_integrator(l, *m)
        e.set_positions(np.stack([s['x']] * K)); e.set_velocities(v0)
        e.set_replica_states(perm)
        e.propagate(77, 3, moves[0][4] if all(m == moves[0] for m in moves) else False)
        out = (e.get_positions(), e.get_velocities(), e.get_replica_energies())
        e.close()
        return out
    xm, vm, (pm, km) = run([A, A, B, B])
    xa, va, (pa, ka) = run([A] * 4)
    xb, vb, (pb, kb) = run([B] * 4)
    for k in range(K):
        x_ref, v_ref, p_ref, k_ref = (xa, va, pa, ka) if perm[k] < 2 else (xb, vb, pb, kb)
        assert np.array_equal(xm[k], x_ref[k]) and np.array_equal(vm[k], v_ref[k]), k
        # (the two kernel instantiations may contract the f64 energy sums differently: last-bit differences)
        assert np.isclose(pm[k], p_ref[k], rtol=1e-12, atol=1e-9) and np.isclose(km[k], k_ref[k], rtol=1e-12, atol=1e-9), k
    assert not np.array_equal(xa[0], xb[0])   # the two moves really differ
