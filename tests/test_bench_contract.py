"""bench.py prints exactly one JSON line on stdout with the contract's keys (checked on the CPU reference arm,
which needs no GPU; the GPU arm shares the line builder).  --dump-outputs is checked on both arms."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), *args], cwd=ROOT, env=e, capture_output=True,
                       text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    return p.stdout


def test_reference_arm_prints_one_json_line_with_contract_keys():
    out = run_bench('--impl', 'reference', '--steps', '1', '--warmup', '0', '--replicas', '8', '--atoms', '64', '--md-steps', '5')
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, out
    d = json.loads(lines[0])
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e', 'impl'):
        assert key in d, key
    assert d['impl'] == 'reference' and d['steps'] == 1 and d['higher_is_better'] is True
    assert d['value'] > 0 and abs(d['value'] - 1000.0 / d['ms_per_step']) < 1e-6 * d['value']
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0 and d['e2e']['value'] == d['value']
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert 'workload' in d['config'] and 'model' not in d['config']


def test_reference_arm_other_ranks_exit_silently():
    out = run_bench('--impl', 'reference', '--gpus', '2', '--steps', '1', '--warmup', '0',
                    env={'RANK': '1', 'WORLD_SIZE': '2', 'LOCAL_RANK': '1'})
    assert out.strip() == ''


def test_config4_reference_arm_keeps_the_contract():
    """--workload config4 (BASELINE configs[3], AlanineDipeptideVacuum T-REMD): the same line, its own metric name."""
    out = run_bench('--workload', 'config4', '--impl', 'reference', '--steps', '1', '--warmup', '0', '--replicas', '4',
                    '--md-steps', '20')
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, out
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and 'AlanineDipeptideVacuum' in d['metric'] and d['config']['atoms'] == 22
    assert d['config']['replicas'] == 4 and d['config']['md_steps'] == 20 and d['value'] > 0
    assert d['cpu_baseline']['kind'] == 'port' and d['e2e']['value'] == d['value']


DUMPED = ('positions', 'velocities', 'energy_thermodynamic_states', 'replica_thermodynamic_states', 'n_accepted_matrix',
          'n_proposed_matrix')


def load_dump(d):
    import numpy as np
    assert sorted(os.listdir(d)) == sorted(n + '.npy' for n in DUMPED)
    out = {n: np.load(os.path.join(d, n + '.npy')) for n in DUMPED}
    assert all(a.dtype == np.float64 for a in out.values())
    return out


def test_reference_arm_dumps_the_last_iteration_and_repeats_it(tmp_path):
    import numpy as np
    args = ('--impl', 'reference', '--steps', '2', '--warmup', '0', '--replicas', '6', '--atoms', '32', '--md-steps', '4')
    run_bench(*args, '--dump-outputs', str(tmp_path / 'a'))
    run_bench(*args, '--dump-outputs', str(tmp_path / 'b'))
    a, b = load_dump(str(tmp_path / 'a')), load_dump(str(tmp_path / 'b'))
    assert a['positions'].shape == (6, 32, 3) and a['energy_thermodynamic_states'].shape == (6, 6)
    assert sorted(a['replica_thermodynamic_states']) == list(range(6)) and a['n_proposed_matrix'].sum() > 0
    for n in DUMPED:
        assert np.array_equal(a[n], b[n]), n


def test_dump_keeps_a_fixed_sample_of_rows_above_the_limit(tmp_path, monkeypatch):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, 'DUMP_LIMIT', 4096)
    big, small = np.arange(1000.0).reshape(200, 5), np.arange(3, dtype=np.int64)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), {'big': big, 'small': small})
    rows = np.load(str(tmp_path / 'a' / 'big_rows.npy'))
    got = np.load(str(tmp_path / 'a' / 'big.npy'))
    assert got.nbytes < 4096 and np.array_equal(got, big[rows.astype(int)]) and np.array_equal(rows, np.sort(rows))
    assert np.array_equal(rows, np.load(str(tmp_path / 'b' / 'big_rows.npy')))
    assert sum(os.path.getsize(str(p)) for p in (tmp_path / 'a').iterdir()) < 4096 + 4 * 128   # + the .npy headers
    assert np.load(str(tmp_path / 'a' / 'small.npy')).dtype == np.float64


@pytest.mark.gpu
def test_device_dump_repeats_and_steps_count_the_timed_iterations(tmp_path):
    """Same arguments, same arrays; and --steps sets how many iterations run: 1 warm-up + 2 timed steps end where
    2 warm-up + 1 timed step end, and not where 1 + 1 end."""
    import numpy as np
    small = ('--replicas', '16', '--atoms', '128', '--md-steps', '20', '--no-e2e', '--no-cpu-baseline')
    runs = {'w1s2': ('1', '2'), 'w1s2_again': ('1', '2'), 'w2s1': ('2', '1'), 'w1s1': ('1', '1')}
    d = {}
    for name, (w, s) in runs.items():
        line = json.loads(run_bench('--warmup', w, '--steps', s, *small, '--dump-outputs', str(tmp_path / name),
                                    env={'RX_BENCH_NO_CLOCKS': '1'}).strip().splitlines()[-1])
        assert line['steps'] == int(s)
        d[name] = load_dump(str(tmp_path / name))
    assert d['w1s2']['positions'].shape == (16, 128, 3)
    for n in DUMPED:
        assert np.array_equal(d['w1s2'][n], d['w1s2_again'][n]), n
        assert np.array_equal(d['w1s2'][n], d['w2s1'][n]), n
    assert not np.array_equal(d['w1s2']['positions'], d['w1s1']['positions'])
