#!/usr/bin/env python
"""bench.py -- replica-exchange iterations/second on the 256-replica alchemical Lennard-Jones fluid.

Workload (BASELINE.json metric, SURVEY.md section 8d config 3): LennardJonesFluid(512) made alchemical with
AbsoluteAlchemicalFactory (atoms 0-9, annihilate_sterics=False, disable_alchemical_dispersion_correction=True),
K = M = 256 states lambda_l = 1 - l/(K-1) at 300 K, LangevinSplittingDynamicsMove("V R O R V", 1 fs, 10/ps,
500 steps), swap-all mixing (K^3 = 16 777 216 attempts).  One "step" = one iteration = mix -> propagate ->
energies (multistatesampler.py:776-782).  Strong scaling: the 256 replicas are sharded over --gpus ranks.

  python bench.py --gpus 1 --steps 5 --warmup 3
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...        (the CPU arm: the oracle port of the reference's path, all host cores)
  python bench.py ... --dump-outputs DIR      (also writes the arrays of the last timed iteration, to compare two builds)

`value`   : device-resident loop (rx_run_iterations), CUDA events on the engine's stream, max over ranks.
`e2e`     : the same iterations through the public API (ReplicaExchangeSampler.run with host_resident_states=True):
            every iteration pushes all positions+velocities from (pinned-staged) host memory, and pulls them, the
            energy matrix, the permutation and the swap statistics back.
torch.distributed (gloo) is plumbing only: barrier, max-reduction of the timings, broadcast of the NCCL id.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

KB = 8.31446261815324e-3


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--replicas', type=int, default=256)
    ap.add_argument('--atoms', type=int, default=512)
    ap.add_argument('--md-steps', type=int, default=500)
    ap.add_argument('--mixing', default='swap-all', choices=['swap-all', 'swap-neighbors', 'none'])
    ap.add_argument('--workload', default='lj', choices=['lj', 'config4'],
                    help="lj: the BASELINE metric's alchemical LJ fluid (default); config4: BASELINE configs[3], T-REMD of "
                         "AlanineDipeptideVacuum (128 temperatures 300-600 K, 1000 steps/iteration; --replicas/--md-steps override)")
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last timed iteration computed (positions, velocities, '
                         'energy matrix, replica -> state map, swap counts) as DIR/<name>.npy in float64')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


# ------------------------------------------------------------------------------------------------------------
def build_workload(K, N):
    from openmmtools_b200 import testsystems, alchemy, states, unit
    fluid = testsystems.LennardJonesFluid(nparticles=N)
    factory = alchemy.AbsoluteAlchemicalFactory(disable_alchemical_dispersion_correction=True)
    region = alchemy.AlchemicalRegion(alchemical_atoms=range(10), annihilate_sterics=False)
    asys = factory.create_alchemical_system(fluid.system, region)
    lambdas = [1.0 - l / (K - 1) for l in range(K)]
    protocol = {'lambda_sterics': lambdas, 'lambda_electrostatics': lambdas}
    tstates = states.create_thermodynamic_state_protocol(
        asys, protocol, constants={'temperature': 300.0 * unit.kelvin},
        composable_states=alchemy.AlchemicalState.from_system(asys))
    sstate = states.SamplerState(fluid.positions, box_vectors=asys.getDefaultPeriodicBoxVectors())
    return fluid, asys, tstates, sstate, lambdas


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md) through NVML in a background
    thread (two light queries per second, plus one at the end of the region).  A polling `nvidia-smi -lms 100` process measurably perturbs this workload
    (it holds driver locks while the host issues the dependent launches of each iteration), so it is only the fallback."""

    def __init__(self, device, period=1.0):
        import threading
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._smi = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(int(device))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._run, args=(period,), daemon=True)
            self._thread.start()
        except Exception:
            self._start_smi(device)

    def _sample(self):
        nv = self.nv
        self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for name, bit in (('hw_slowdown', 0x8), ('sw_power_cap', 0x4), ('sw_thermal_slowdown', 0x20),
                          ('hw_thermal_slowdown', 0x40)):
            if r & bit:
                self.reasons.add(name)

    def _run(self, period):
        while not self._stop.is_set():
            try:
                self._sample()
            except Exception:
                pass
            self._stop.wait(period)

    def _start_smi(self, device):
        q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        self.path = '/tmp/rx_clocks_%d.csv' % os.getpid()
        try:
            self.f = open(self.path, 'w')
            self._smi = subprocess.Popen(['nvidia-smi', '-i', str(device), '--query-gpu=' + q, '--format=csv,noheader,nounits',
                                          '-lms', '500'], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self._smi = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'source': None}
        if self._thread is not None:
            try:
                self._sample()      # at least one sample inside the region even for very short runs
            except Exception:
                pass
            self._stop.set()
            self._thread.join(timeout=2)
            if self.samples:
                out = {'sm_mhz': float(np.median(self.samples)), 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                       'samples': len(self.samples), 'source': 'nvml thread, 1 s period'}
            return out
        if self._smi is None:
            return out
        self._smi.terminate()
        try:
            self._smi.wait(timeout=5)
        except Exception:
            self._smi.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            c = [x.strip() for x in line.split(',')]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), c[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if sm:
            out = {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                   'samples': len(sm), 'source': 'nvidia-smi -lms 500'}
        return out


class Dist:
    def __init__(self, world):
        self.world = world
        self.rank = int(os.environ.get('RANK', '0'))
        self.dist = None
        if world > 1:
            import torch.distributed as dist
            os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
            os.environ.setdefault('MASTER_PORT', '29511')
            dist.init_process_group('gloo', rank=self.rank, world_size=world)
            self.dist = dist

    def barrier(self):
        if self.dist:
            self.dist.barrier()

    def max(self, v):
        if not self.dist:
            return v
        import torch
        t = torch.tensor([v], dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0])

    def sum(self, v):
        if not self.dist:
            return v
        import torch
        t = torch.tensor([v], dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t[0])


DUMP_LIMIT = 64 << 20      # bytes written by --dump-outputs at most


def dump_outputs(path, arrays):
    """--dump-outputs: each array as <path>/<name>.npy in float64 (the integer maps and counts are exact there).  Above
    DUMP_LIMIT bytes in all, each array keeps a fixed, seeded sample of its rows and <name>_rows.npy lists them."""
    arrays = {k: np.asarray(v, np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    with_rows = total + sum(8 * a.shape[0] for a in arrays.values() if a.ndim)     # each kept row costs 8 more bytes
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_LIMIT and a.ndim and a.shape[0] > 1:
            n = max(1, int(a.shape[0] * 0.9 * DUMP_LIMIT / with_rows))
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], n, replace=False))
            np.save(os.path.join(path, name + '_rows.npy'), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(path, name + '.npy'), a)


def engine_outputs(eng, dist):
    """What the device-resident loop leaves for its caller after its last iteration; the replicas of every rank."""
    def all_replicas(local):
        full = np.zeros((eng.K,) + local.shape[1:])
        full[eng.k0:eng.k1] = local
        if dist.dist:
            import torch
            t = torch.from_numpy(full)
            dist.dist.all_reduce(t, op=dist.dist.ReduceOp.SUM)
            full = t.numpy()
        return full
    nacc, nprop = eng.get_mix_counts()
    return {'positions': all_replicas(eng.get_positions()), 'velocities': all_replicas(eng.get_velocities()),
            'energy_thermodynamic_states': eng.get_energies(), 'replica_thermodynamic_states': eng.get_replica_states(),
            'n_accepted_matrix': nacc, 'n_proposed_matrix': nprop}


# ------------------------------------------------------------------------------------------------------------
def cpu_arm(args, steps, warmup, full_line):
    """The reference's CPU path restated (oracle/rx_oracle.c): numba-identical mixing (single thread, it is a
    serial chain), Verlet-list Langevin propagation and the energy matrix with OpenMP over replicas on all host
    cores.  One step = one full iteration of the same workload."""
    os.environ.setdefault('OMP_PROC_BIND', 'true')     # pinned threads: a repeatable CPU arm (read when libgomp starts)
    os.environ.setdefault('OMP_PLACES', 'threads')
    from oracle import oracle
    K, N = args.replicas, args.atoms
    fluid, asys, tstates, sstate, lambdas = build_workload(K, N)
    L = asys.box_vectors[0, 0]
    osys = oracle.LJSystem(asys.sigma, asys.epsilon, asys.masses, asys.alchemical_mask(), (L, L, L), asys.cutoff,
                           asys.switching_distance, use_switch=True)
    # every host core this process may run on, whatever OMP_NUM_THREADS says (torchrun exports OMP_NUM_THREADS=1)
    threads = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    rng = np.random.default_rng(2024)
    x = np.stack([np.asarray(sstate._positions)] * K)
    v = rng.normal(scale=np.sqrt(KB * 300.0 / asys.masses[0]), size=x.shape)
    lam = np.array(lambdas); betas = np.full(K, 1.0 / (KB * 300.0)); kTs = np.full(K, KB * 300.0)
    perm = np.arange(K, dtype=np.int64)
    mt = oracle.MT(1234)
    u = osys.energy_matrix(x, lam, betas, None, threads)
    times = []
    for it in range(warmup + steps):
        t0 = time.time()
        nacc = np.zeros((K, K), np.int64); nprop = np.zeros((K, K), np.int64)
        if args.mixing == 'swap-all':
            oracle.mix_swap_all(mt, K ** 3, perm, u, nacc, nprop)
        elif args.mixing == 'swap-neighbors':
            oracle.mix_swap_neighbors(mt, perm, u, nacc, nprop)
        t1 = time.time()
        osys.propagate_replicas(x, v, lam[perm], kTs, 0.001, 10.0, args.md_steps, 7 + it, threads)
        t2 = time.time()
        u = osys.energy_matrix(x, lam, betas, None, threads)
        t3 = time.time()
        if it >= warmup:
            times.append((t3 - t0, t1 - t0, t2 - t1, t3 - t2))
    if full_line and args.dump_outputs:
        dump_outputs(args.dump_outputs, {'positions': x, 'velocities': v, 'energy_thermodynamic_states': u,
                                         'replica_thermodynamic_states': perm, 'n_accepted_matrix': nacc,
                                         'n_proposed_matrix': nprop})
    tt = np.array(times)
    mean = tt[:, 0].mean()
    base = {'value': 1.0 / mean, 'unit': 'iterations/s', 'cores': threads, 'kind': 'port',
            'sample': '%d full iterations (K=%d, N=%d, %d BAOAB steps, %s): mixing single-threaded (serial chain), '
                      'propagation+energies OpenMP over replicas on %d threads; oracle/rx_oracle.c (OpenMM itself is '
                      'not installable here)' % (steps, K, N, args.md_steps, args.mixing, threads),
            'phases_ms': {'mix': 1e3 * tt[:, 1].mean(), 'propagate': 1e3 * tt[:, 2].mean(), 'energies': 1e3 * tt[:, 3].mean()}}
    if not full_line:
        return base
    line = {'impl': 'reference', 'metric': 'replica-exchange iterations/sec, 256-replica alchemical LJ fluid',
            'value': 1.0 / mean, 'unit': 'iterations/s', 'n_gpus': args.gpus, 'steps': steps, 'warmup': warmup,
            'ms_per_step': 1e3 * mean, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
            'dtype': 'f64', 'data': 'synthetic',
            'config': workload_config(args), 'cpu_baseline': base,
            'e2e': {'value': 1.0 / mean, 'unit': 'iterations/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    return line


def workload_config(args):
    std = args.atoms == 512 and args.md_steps == 500 and args.mixing == 'swap-all'
    label = {64: 'configs[1]', 256: 'configs[2]'}.get(args.replicas) if std else None
    return {'workload': '%s: alchemical LennardJonesFluid(%d), %d lambda-replicas, %d BAOAB steps/iter, %s'
                        % (label or 'non-BASELINE variant', args.atoms, args.replicas, args.md_steps, args.mixing),
            'replicas': args.replicas, 'atoms': args.atoms, 'md_steps': args.md_steps, 'mixing': args.mixing,
            'parallelism': 'replica-sharded x%d, NCCL allgather of energy rows, replicated mixing' % args.gpus,
            'l2': 'no explicit flush: each iteration streams ~0.8 GB of RNG words + slot records (> 126 MB L2); the '
                  '4 MB replica state is the resident working set by design'}


def state_digest(sampler, dist):
    """A digest of the trajectory that must not depend on the number of GPUs: CRC32 of every replica's positions (each rank
    contributes the replicas it owns), of the replica -> state map and of the energy matrix, after all timed work."""
    import zlib
    e = sampler._engine
    K = sampler.n_replicas
    x = e.get_positions()
    crc = np.zeros(K, np.float64)
    for r, k in enumerate(range(e.k0, e.k1)):
        crc[k] = float(zlib.crc32(np.ascontiguousarray(x[r]).tobytes()))
    if dist.dist:
        import torch
        t = torch.from_numpy(crc)
        dist.dist.all_reduce(t, op=dist.dist.ReduceOp.SUM)
        crc = t.numpy()
    perm = np.asarray(sampler._engine.get_replica_states(), np.int64)
    u = e.get_energies()
    return {'positions': '%08x' % zlib.crc32(crc.astype(np.uint64).tobytes()), 'replica_states': '%08x' % zlib.crc32(perm.tobytes()),
            'energies': '%08x' % zlib.crc32(np.ascontiguousarray(u).tobytes()),
            'note': 'after warm-up + timed + end-to-end iterations; equal digests at every --gpus = the same trajectory'}


# ------------------------------------------------------------------------------------------------------------
# BASELINE configs[3] with the same contract (not the default: the headline metric is the LJ fluid)
C4_METRIC = 'replica-exchange iterations/sec, AlanineDipeptideVacuum T-REMD (BASELINE configs[3])'


def config4_sizes(args):
    K = 128 if args.replicas == 256 else args.replicas          # (256 / 500 are the LJ defaults of the flags)
    n_steps = 1000 if args.md_steps == 500 else args.md_steps
    return K, n_steps


def config4_config(args, K, n_steps):
    return {'workload': '%s: testsystems.AlanineDipeptideVacuum (22 atoms, HBonds constraints, no cutoff), ParallelTemperingSampler, %d '
                        'temperatures 300-600 K, %d steps of 2 fs per iteration (V R O R V, 5/ps), swap-all'
                        % ('configs[3]' if (K, n_steps) == (128, 1000) else 'non-BASELINE variant of configs[3]', K, n_steps),
            'replicas': K, 'atoms': 22, 'md_steps': n_steps, 'mixing': 'swap-all',
            'parallelism': 'replica-sharded x%d, NCCL allgather of energy rows, replicated mixing' % args.gpus,
            'l2': 'no explicit flush: each iteration streams the RNG words and slot records of K^3 swap attempts (> 126 MB L2 '
                  'from K = 128 on); the replica state (K x 22 atoms) is the resident working set by design'}


def cpu_arm_config4(args, steps, warmup, full_line):
    """The reference's CPU path for configs[3] restated (oracle/rx_oracle_mol.c + rx_oracle.c): constrained Langevin
    dynamics per replica (one host thread per replica through a thread pool: the C calls release the GIL), K x K
    reduced-potential matrix, numba-identical swap-all mixing on one thread."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle
    from openmmtools_b200 import testsystems, unit
    K, n_steps = config4_sizes(args)
    a = testsystems.AlanineDipeptideVacuum()
    m = oracle.Molecule(a.system)
    x0 = np.ascontiguousarray(a.positions.value_in_unit(unit.nanometer), np.float64)
    T = np.logspace(np.log10(300.0), np.log10(600.0), num=K)      # paralleltempering.py:162
    betas = 1.0 / (KB * T)
    threads = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    rng = np.random.default_rng(2024)
    xs = [x0.copy() for _ in range(K)]
    vs = [np.ascontiguousarray(rng.normal(size=x0.shape) * np.sqrt(KB * 300.0 / m.mass)[:, None]) for _ in range(K)]
    perm = np.arange(K, dtype=np.int64)
    mt = oracle.MT(1234)
    pool = ThreadPoolExecutor(max_workers=min(threads, K))

    def energies():
        U = np.array(list(pool.map(lambda k: m.energy(xs[k]), range(K))))
        return np.ascontiguousarray(U[:, None] * betas[None, :])

    def step_replica(k_it):
        k, it = k_it
        noise = np.random.default_rng(1000003 * it + k).normal(size=(n_steps, 22, 3))
        m.langevin(xs[k], vs[k], noise, KB * T[perm[k]], 0.002, 5.0, n_steps, 'VRORV', tol=1e-8)

    u = energies()
    times = []
    for it in range(warmup + steps):
        t0 = time.time()
        nacc = np.zeros((K, K), np.int64); nprop = np.zeros((K, K), np.int64)
        oracle.mix_swap_all(mt, K ** 3, perm, u, nacc, nprop)
        t1 = time.time()
        list(pool.map(step_replica, [(k, it) for k in range(K)]))
        t2 = time.time()
        u = energies()
        t3 = time.time()
        if it >= warmup:
            times.append((t3 - t0, t1 - t0, t2 - t1, t3 - t2))
    pool.shutdown()
    if full_line and args.dump_outputs:
        dump_outputs(args.dump_outputs, {'positions': np.stack(xs), 'velocities': np.stack(vs),
                                         'energy_thermodynamic_states': u, 'replica_thermodynamic_states': perm,
                                         'n_accepted_matrix': nacc, 'n_proposed_matrix': nprop})
    tt = np.array(times)
    mean = tt[:, 0].mean()
    base = {'value': 1.0 / mean, 'unit': 'iterations/s', 'cores': min(threads, K), 'kind': 'port',
            'sample': '%d full iterations (K=%d, 22 atoms, %d constrained Langevin steps, swap-all): mixing single-threaded '
                      '(serial chain), one replica per host thread on %d threads (noise drawn by numpy inside the timed region, '
                      'as OpenMM draws its own); oracle/rx_oracle_mol.c + rx_oracle.c (OpenMM itself is not installable here)'
                      % (steps, K, n_steps, min(threads, K)),
            'phases_ms': {'mix': 1e3 * tt[:, 1].mean(), 'propagate': 1e3 * tt[:, 2].mean(), 'energies': 1e3 * tt[:, 3].mean()}}
    if not full_line:
        return base
    return {'impl': 'reference', 'metric': C4_METRIC, 'value': 1.0 / mean, 'unit': 'iterations/s', 'n_gpus': args.gpus,
            'steps': steps, 'warmup': warmup, 'ms_per_step': 1e3 * mean, 'higher_is_better': True, 'scaling': 'strong',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'config': config4_config(args, K, n_steps),
            'cpu_baseline': base,
            'e2e': {'value': 1.0 / mean, 'unit': 'iterations/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}


def main_config4(args, world, rank):
    if args.impl == 'reference':
        if rank == 0:
            _emit(cpu_arm_config4(args, args.steps, max(args.warmup, 0), True))
        return 0
    if world != args.gpus and world > 1:
        raise SystemExit('--gpus %d but WORLD_SIZE=%d' % (args.gpus, world))
    dist = Dist(world)
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    os.environ['LOCAL_RANK'] = str(local_rank)
    from openmmtools_b200 import testsystems, states, mcmc, multistate, unit
    from openmmtools_b200._dist import TorchCommunicator
    K, n_steps = config4_sizes(args)
    a = testsystems.AlanineDipeptideVacuum()
    ts = states.ThermodynamicState(a.system, 300.0 * unit.kelvin)
    move = mcmc.LangevinSplittingDynamicsMove(timestep=2.0 * unit.femtosecond, collision_rate=5.0 / unit.picosecond, n_steps=n_steps)
    comm = TorchCommunicator() if world > 1 else None
    sampler = multistate.ParallelTemperingSampler(mcmc_moves=move, number_of_iterations=10 ** 9, seed=1234, communicator=comm)
    sampler.create(ts, [states.SamplerState(a.positions)], storage=None, min_temperature=300.0 * unit.kelvin,
                   max_temperature=600.0 * unit.kelvin, n_temperatures=K)
    eng = sampler._engine
    sampler._compute_energies()
    eng.run_iterations(args.warmup, 'swap-all', sampler._seed, 1)
    eng.phase_times(reset=True)
    clocks = ClockSampler(local_rank) if (rank == 0 and not os.environ.get('RX_BENCH_NO_CLOCKS')) else None
    dist.barrier()
    eng.timer_mark(0)
    t0 = time.time()
    eng.run_iterations(args.steps, 'swap-all', sampler._seed, 1 + args.warmup)
    eng.timer_mark(1)
    ms = dist.max(eng.timer_elapsed_ms())
    wall = time.time() - t0
    dist.barrier()
    ck = clocks.stop() if clocks else None
    pt = eng.phase_times()
    mstats = eng.mix_stats()
    launches = dist.sum(pt['launches'])
    if args.dump_outputs:
        outputs = engine_outputs(eng, dist)
        if rank == 0:
            dump_outputs(args.dump_outputs, outputs)
    ms_iter = ms / args.steps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    kloc = eng.k1 - eng.k0
    b_prop = kloc * 22 * n_steps * 96.0          # x, v (f64) read + written per atom-step: the streaming model of SURVEY 8(d)
    t_prop = pt['propagate_ms'] / args.steps * 1e-3
    ach = b_prop / t_prop / 1e9 if t_prop > 0 else 0.0
    roof = {'kernel': 'k_propagate_mol', 'bound': 'hbm', 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak,
            'traffic': 284416.0 * kloc / 128.0,
            'traffic_source': 'dram__bytes_read+write of one launch in the committed ncu capture profiles/mol_r2c.summary.txt '
                              '(128 replicas), scaled by replicas per GPU; NOT measured in this run',
            'peak_source': 'MEASURED_PEAKS.json (of measured)' if peaks else 'fallback 6650 GB/s',
            'algorithmic_bytes_per_launch': b_prop, 'share_of_step': pt['propagate_ms'] / args.steps / ms_iter,
            'note': 'one block of four warps per replica, the state on chip for all steps: a latency chain of ~14 k cycles per '
                    'constrained step (DESIGN.md 7, f-2), neither HBM nor FP throughput; the streaming-model figure is given '
                    'for the contract only',
            'dominant_kernel': {'name': 'k_mix_walk2 (+ k_mix_walk_pow2 tail)' if (K & (K - 1)) == 0 else 'k_mix_walk2c',
                                'share_of_step': mstats['walker_ms'] / ms_iter,
                                'bound': 'latency: one warp, one dependent chain per speculation round (exact swap-all chain)',
                                'rounds': mstats['rounds'], 'ns_per_round': 1e6 * mstats['walker_ms'] / max(mstats['rounds'], 1),
                                'attempts_per_round': (K ** 3) / max(mstats['rounds'], 1), 'mix_phase_ms': pt['mix_ms'] / args.steps}}
    e2e = None
    if not args.no_e2e:
        sampler.host_resident_states = True
        sampler._states_stale = True
        sampler._sync_sampler_states()
        sampler._iteration = 1 + args.warmup + args.steps
        n_e2e = max(2, min(args.steps, 10))
        sampler.run(1)
        dist.barrier()
        t0 = time.time()
        sampler.run(n_e2e)
        dt = dist.max(time.time() - t0)
        dist.barrier()
        h2d = kloc * 22 * 3 * 8 * 2
        d2h = kloc * 22 * 3 * 8 * 2 + K * K * 8 + K * 8 + 2 * K * K * 8 + 2 * K * 8
        e2e = {'value': n_e2e / dt, 'unit': 'iterations/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
               'iterations': n_e2e, 'api': 'ParallelTemperingSampler.run(host_resident_states=True)'}
    digest = state_digest(sampler, dist)
    if rank != 0:
        return 0
    line = {'metric': C4_METRIC, 'value': args.steps / (ms * 1e-3), 'unit': 'iterations/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_iter, 'higher_is_better': True, 'scaling': 'strong',
            'vs_baseline': None, 'dtype': 'f32 forces, f64 positions/velocities/constraints/energies/mixing', 'data': 'synthetic',
            'config': config4_config(args, K, n_steps), 'roofline': roof,
            'phases_ms': {'mix': pt['mix_ms'] / args.steps, 'propagate': pt['propagate_ms'] / args.steps,
                          'energies_incl_allgather': pt['energies_ms'] / args.steps},
            'mixing_stats': mstats, 'clocks': ck, 'e2e': e2e, 'gpu_launches': int(launches), 'state_digest': digest,
            'host_wall_ms_per_step': 1e3 * wall / args.steps}
    if not args.no_cpu_baseline:
        try:
            line['cpu_baseline'] = cpu_arm_config4(args, 2, 1, False)
        except Exception as e:
            line['cpu_baseline'] = {'error': repr(e)}
    _emit(line)
    return 0


_REAL_STDOUT = sys.stdout


# ------------------------------------------------------------------------------------------------------------
def _emit(line):
    """The one JSON line of the contract, on the process's ORIGINAL stdout."""
    _REAL_STDOUT.write(json.dumps(line) + '\n')
    _REAL_STDOUT.flush()


def main():
    # Native libraries may write to file descriptor 1 (NCCL prints its version banner there when NCCL_DEBUG is set):
    # keep the original stdout for the JSON line only and point fd 1 at stderr for everything else.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)
    args = parse()
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    if args.workload == 'config4':
        return main_config4(args, world, rank)
    if args.impl == 'reference':
        if rank != 0:
            return 0
        line = cpu_arm(args, args.steps, max(args.warmup, 0), True)
        _emit(line)
        return 0

    if world != args.gpus and world > 1:
        raise SystemExit('--gpus %d but WORLD_SIZE=%d' % (args.gpus, world))
    dist = Dist(world)
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    K, N = args.replicas, args.atoms
    from openmmtools_b200 import multistate, mcmc, unit, _lib
    from openmmtools_b200._dist import TorchCommunicator
    fluid, asys, tstates, sstate, lambdas = build_workload(K, N)
    mixing = None if args.mixing == 'none' else args.mixing
    move = mcmc.LangevinSplittingDynamicsMove(timestep=1.0 * unit.femtosecond, collision_rate=10.0 / unit.picosecond,
                                              n_steps=args.md_steps, reassign_velocities=False, splitting='V R O R V')
    comm = TorchCommunicator() if world > 1 else None
    os.environ['LOCAL_RANK'] = str(local_rank)
    sampler = multistate.ReplicaExchangeSampler(mcmc_moves=move, number_of_iterations=10 ** 9, replica_mixing_scheme=mixing,
                                                seed=1234, communicator=comm)
    sampler.create(tstates, [sstate], storage=None)
    eng = sampler._engine
    # iteration 0 energies, as run() does
    sampler._compute_energies()

    # ---------------- device-resident loop
    eng.run_iterations(args.warmup, mixing, sampler._seed, 1)
    eng.phase_times(reset=True)
    clocks = ClockSampler(local_rank) if (rank == 0 and not os.environ.get('RX_BENCH_NO_CLOCKS')) else None
    dist.barrier()
    eng.timer_mark(0)
    t0 = time.time()
    eng.run_iterations(args.steps, mixing, sampler._seed, 1 + args.warmup)
    eng.timer_mark(1)
    ms_dev = eng.timer_elapsed_ms()
    wall = time.time() - t0
    dist.barrier()
    ms = dist.max(ms_dev)
    ck = clocks.stop() if clocks else None
    pt = eng.phase_times()
    mstats = eng.mix_stats()
    launches = dist.sum(pt['launches'])
    if args.dump_outputs:
        outputs = engine_outputs(eng, dist)
        if rank == 0:
            dump_outputs(args.dump_outputs, outputs)
    value = args.steps / (ms * 1e-3)

    # roofline of k_propagate (the HBM-streaming kernel of SURVEY.md 8d): algorithmic bytes per launch
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    kloc = eng.k1 - eng.k0
    b_prop = kloc * N * args.md_steps * 64.0
    t_prop = pt['propagate_ms'] / max(args.steps, 1) * 1e-3
    ach = b_prop / t_prop / 1e9 if t_prop > 0 else 0.0
    b_iter = K * N * args.md_steps * 64.0 / world + K * N * 16.0 / world + 2 * K * K * 8.0 + K * 8.0
    traffic = None
    tj = {}
    try:    # dram__bytes_read.sum + dram__bytes_write.sum of one launch from the committed ncu capture (K=256 on one GPU)
        tj = json.load(open(os.path.join(ROOT, 'profiles', 'k_propagate_traffic.json')))
        traffic = (tj['dram_bytes_read'] + tj['dram_bytes_write']) * (kloc / 256.0)
    except Exception:
        pass
    ms_iter = ms / args.steps
    t_mix = pt['mix_ms'] / max(args.steps, 1)
    issue = None
    try:    # instruction-issue roofline of k_propagate: warp instructions of one launch from the same committed capture
        winst = tj['warp_instructions'] * (kloc / 256.0) * (args.md_steps / 500.0)
        sm_hz = (ck or {}).get('sm_mhz') or 1965.0
        peak_ipc = 148 * 4 * sm_hz * 1e6
        issue = {'warp_instructions_per_launch': winst, 'peak_warp_instructions_per_s': peak_ipc,
                 'frac': winst / t_prop / peak_ipc if t_prop > 0 else None,
                 'source': 'smsp__inst_executed.sum of profiles/k_propagate_traffic.json (ncu capture, K=256, 500 steps), '
                           'scaled by replicas and steps; 148 SMs x 4 issue slots x the SM clock sampled in this run'}
    except Exception:
        pass
    roof = {'kernel': 'k_propagate', 'bound': 'hbm', 'achieved': ach, 'peak': peak, 'unit': 'GB/s',
            'frac': ach / peak, 'traffic': traffic,
            'traffic_source': 'dram__bytes_read+write of one launch in the committed ncu capture profiles/k_propagate_traffic.json '
                              '(K=256), scaled by replicas per GPU; NOT measured in this run',
            'peak_source': 'MEASURED_PEAKS.json (of measured)' if peaks else 'fallback 6650 GB/s',
            'algorithmic_bytes_per_launch': b_prop,
            'share_of_step': pt['propagate_ms'] / max(args.steps, 1) / ms_iter,
            'issue_roofline': issue,
            'note': 'the streaming model of SURVEY.md 8(d) (x, v read + written per atom-step); the state stays on chip for '
                    'all steps, so real DRAM traffic is `traffic` and the kernel is instruction-issue bound: see issue_roofline',
            'whole_iteration': {'bytes': b_iter, 'achieved': b_iter / (ms_iter * 1e-3) / 1e9,
                                'frac': b_iter / (ms_iter * 1e-3) / 1e9 / peak},
            'dominant_kernel': {
                'name': 'k_mix_walk2 (+ k_mix_walk_pow2 tail)' if mixing == 'swap-all' else 'k_propagate',
                'share_of_step': (mstats['walker_ms'] / ms_iter) if mixing == 'swap-all' else pt['propagate_ms'] / max(args.steps, 1) / ms_iter,
                'bound': 'latency: one warp, one dependent chain per speculation round (exact swap-all chain); neither '
                         'HBM nor FP throughput' if mixing == 'swap-all' else 'instruction issue',
                'rounds': mstats['rounds'], 'ns_per_round': 1e6 * mstats['walker_ms'] / max(mstats['rounds'], 1),
                'attempts_per_round': (K ** 3) / max(mstats['rounds'], 1) if mixing == 'swap-all' else None,
                'mix_phase_ms': t_mix}}

    # ---------------- end to end through the public API with host-resident sampler states
    e2e = None
    if not args.no_e2e:
        sampler.host_resident_states = True
        sampler._states_stale = True
        sampler._sync_sampler_states()
        sampler._iteration = 1 + args.warmup + args.steps
        n_e2e = max(2, min(args.steps, 5))
        sampler.run(1)      # warm the host path
        dist.barrier()
        t0 = time.time()
        sampler.run(n_e2e)
        dt = time.time() - t0
        dist.barrier()
        dt = dist.max(dt)
        h2d = kloc * N * 3 * 8 * 2
        d2h = kloc * N * 3 * 8 * 2 + K * K * 8 + K * 8 + 2 * K * K * 8 + 2 * K * 8
        e2e = {'value': n_e2e / dt, 'unit': 'iterations/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
               'iterations': n_e2e, 'api': 'ReplicaExchangeSampler.run(host_resident_states=True)'}

    digest = state_digest(sampler, dist)
    if rank != 0:
        return 0
    line = {'metric': 'replica-exchange iterations/sec, 256-replica alchemical LJ fluid',
            'value': value, 'unit': 'iterations/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
            'dtype': 'f32 dynamics, f64 energies and mixing', 'data': 'synthetic',
            'config': workload_config(args), 'roofline': roof,
            'phases_ms': {'mix': pt['mix_ms'] / args.steps, 'propagate': pt['propagate_ms'] / args.steps,
                          'energies_incl_allgather': pt['energies_ms'] / args.steps},
            'mixing_stats': mstats, 'clocks': ck, 'e2e': e2e, 'gpu_launches': int(launches), 'state_digest': digest,
            'host_wall_ms_per_step': 1e3 * wall / args.steps}
    if not args.no_cpu_baseline:
        try:
            line['cpu_baseline'] = cpu_arm(args, 2, 1, False)
        except Exception as e:   # the oracle is test infrastructure; never fail the GPU number because of it
            line['cpu_baseline'] = {'error': repr(e)}
    _emit(line)
    return 0


if __name__ == '__main__':
    sys.exit(main())
