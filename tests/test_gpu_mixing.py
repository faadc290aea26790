"""GPU mixing kernels (through the C ABI) against the golden vectors of the real reference and, at full
size, against the pinned CPU oracle.  Bit-exact: permutation and both count matrices."""
import os
import numpy as np
import pytest
from energy_models import energies
from helpers import gpu_engine

pytestmark = pytest.mark.gpu
G = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'mixing_golden.npz'))


def digest(mat):
    m = mat.astype(np.uint64).ravel()
    w = (np.arange(m.size, dtype=np.uint64) * np.uint64(2654435761) + np.uint64(1))
    return np.array([m.sum(), (m * m).sum(), (m * w).sum()], dtype=np.uint64)


def check_counts(key, mat):
    if mat.shape[0] >= 100:
        assert np.array_equal(G[key + '_digest'], digest(mat)), key
    else:
        assert np.array_equal(G[key], mat), key


def parse(tag):
    _, K, s, model = tag.split('_')
    return int(K[1:]), int(s[1:]), model


@pytest.mark.parametrize('tag', [str(t) for t in G['all_cases']])
def test_swap_all_golden(tag):
    K, seed, model = parse(tag)
    u = energies(model, K, K * 1000 + (seed % 1000))
    e = gpu_engine(0, K, K)
    e.set_energies(u)
    e.set_replica_states(np.arange(K))
    e.mix_seed(seed, 0)
    for call, nswap in ((1, K ** 3), (2, K ** 3), (3, 777)):
        st, nacc, nprop = e.mix_swap_all(nswap)
        assert np.array_equal(st, G[f'{tag}_perm{call}']), (tag, call)
        check_counts(f'{tag}_nacc{call}', nacc)
        check_counts(f'{tag}_nprop{call}', nprop)
    e.close()


@pytest.mark.parametrize('tag', [str(t) for t in G['nbr_cases']])
def test_swap_neighbors_golden(tag):
    K, seed, model = parse(tag)
    u = energies(model, K, K * 77 + seed % 1000)
    e = gpu_engine(0, K, K)
    e.set_energies(u)
    e.set_replica_states(np.arange(K))
    e.mix_seed(seed, 1)
    for it in range(6):
        st, nacc, nprop = e.mix_swap_neighbors()
        assert np.array_equal(st, G[f'{tag}_perms'][it]), (tag, it)
    check_counts(f'{tag}_nacc_last', nacc)
    check_counts(f'{tag}_nprop_last', nprop)
    e.close()


@pytest.mark.parametrize('K,model,seed', [(256, 'flat', 5), (256, 'normal', 6), (256, 'zeros', 7), (512, 'ladder', 8),
                                          (1, 'zeros', 1), (96, 'flat', 9)])
def test_swap_all_full_size_vs_oracle(K, model, seed):
    """BASELINE.json sizes (K=256: 16.7M attempts) and beyond, three consecutive iterations, against the CPU
    oracle that test_oracle_mixing.py pins to the reference."""
    from oracle import oracle
    u = energies(model, K, 4242 + K)
    e = gpu_engine(0, K, K)
    e.set_energies(u)
    e.set_replica_states(np.arange(K))
    e.mix_seed(seed, 0)
    mt = oracle.MT(seed)
    st_o = np.arange(K, dtype=np.int64)
    nswap = K ** 3 if K <= 256 else 3_000_000
    for it in range(2):
        st, nacc, nprop = e.mix_swap_all(nswap)
        na = np.zeros((K, K), np.int64); npr = np.zeros((K, K), np.int64)
        oracle.mix_swap_all(mt, nswap, st_o, u, na, npr)
        assert np.array_equal(st, st_o)
        assert np.array_equal(nacc, na) and np.array_equal(nprop, npr)
        assert nprop.sum() == 2 * nswap
        assert sorted(st) == list(range(K))
    e.close()


@pytest.mark.parametrize('K,model,nswap,seed', [(3, 'flat', 200_000, 31), (5, 'normal', 200_000, 32), (12, 'flat', 300_000, 33),
                                                (65, 'flat', 65 ** 3, 34), (100, 'normal', 100 ** 3, 35),
                                                (127, 'ladder', 500_000, 36), (129, 'normal', 500_000, 37),
                                                (200, 'normal', 2_000_000, 38), (257, 'normal', 300_000, 40),
                                                (300, 'flat', 300_000, 41), (383, 'ladder', 300_000, 42),
                                                (600, 'ladder', 1_000_000, 43), (767, 'normal', 300_000, 44),
                                                (1000, 'flat', 1_000_000, 39), (2047, 'normal', 300_000, 45)])
@pytest.mark.parametrize('path', ['default', 'serial'])
def test_swap_all_any_k_vs_oracle(monkeypatch, K, model, nswap, seed, path):
    """K that is not a power of two.  default: the walk2 organisation in candidate coordinates (k_mix_walk2c, K < 256) or the
    walker over word positions (k_mix_walk_any, 257 <= K <= 4095), each followed by the plain loop for the end of a pass;
    with RX_WALK_SERIAL=1 the plain loop alone; three iterations each."""
    from oracle import oracle
    serial = path == 'serial'
    if serial:
        if nswap > 300_000: pytest.skip('the plain loop takes 0.6 us per attempt')
        monkeypatch.setenv('RX_WALK_SERIAL', '1')
    u = energies(model, K, 777 + K)
    e = gpu_engine(0, K, K)
    e.set_energies(u)
    e.set_replica_states(np.arange(K))
    e.mix_seed(seed, 0)
    mt = oracle.MT(seed)
    st_o = np.arange(K, dtype=np.int64)
    for it in range(3):
        st, nacc, nprop = e.mix_swap_all(nswap)
        na = np.zeros((K, K), np.int64); npr = np.zeros((K, K), np.int64)
        oracle.mix_swap_all(mt, nswap, st_o, u, na, npr)
        assert np.array_equal(st, st_o), it
        assert np.array_equal(nacc, na) and np.array_equal(nprop, npr), it
    stats = e.mix_stats()
    if serial:
        assert stats['rounds'] == 0
    else:
        assert 0 < stats['rounds'] < nswap   # the walker ran and committed several attempts per round
    # the stream position: the next word both generators produce is the same one
    e2 = gpu_engine(0, K, K); e2.mix_seed(seed, 0); e2.mix_skip(e.mix_stream_position(0), 0)
    e2.set_energies(u); e2.set_replica_states(np.arange(K))
    st2, _, _ = e2.mix_swap_all(1000)
    st_o2 = np.arange(K, dtype=np.int64)
    oracle.mix_swap_all(mt, 1000, st_o2, u, np.zeros((K, K), np.int64), np.zeros((K, K), np.int64))
    assert np.array_equal(st2, st_o2)
    e2.close()
    e.close()


@pytest.mark.parametrize('K,kind', [(100, 'equal_rows'), (100, 'nonfinite'), (37, 'equal_rows'), (300, 'equal_rows'),
                                    (300, 'nonfinite')])
def test_swap_all_any_k_hard_matrices(K, kind):
    """Identical rows (iteration 0 of a run whose replicas start from one configuration: every log_p is a rounding error
    around 0) and non-finite entries."""
    from oracle import oracle
    rng = np.random.default_rng(5)
    if kind == 'equal_rows':
        u = np.tile(rng.normal(0, 30, K)[None, :], (K, 1))
    else:
        u = rng.normal(0, 3, (K, K)); u[3, 5] = np.inf; u[7, :] = np.nan; u[11, 2] = -np.inf; u[20, 20] = 1e300
    u = np.ascontiguousarray(u)
    nswap = 200_000
    e = gpu_engine(0, K, K)
    e.set_energies(u); e.set_replica_states(np.arange(K)); e.mix_seed(77, 0)
    mt = oracle.MT(77); st_o = np.arange(K, dtype=np.int64)
    with np.errstate(all='ignore'):
        for it in range(2):
            st, nacc, nprop = e.mix_swap_all(nswap)
            na = np.zeros((K, K), np.int64); npr = np.zeros((K, K), np.int64)
            oracle.mix_swap_all(mt, nswap, st_o, u, na, npr)
            assert np.array_equal(st, st_o), (kind, it)
            assert np.array_equal(nacc, na) and np.array_equal(nprop, npr), (kind, it)
    e.close()


def _exp_correctly_rounded(x):
    """exp(x) rounded to nearest from 60-digit arithmetic (float(Decimal) rounds correctly)."""
    from decimal import Decimal, getcontext
    getcontext().prec = 60
    return float(Decimal(float(x)).exp())


def _libm_decides_like_exact_arithmetic(U, lp):
    """The reference's test U < exp(lp) with the host libm's exp against the same test with the correctly rounded exp.  They
    differ only where the libm is not correctly rounded AND U is the neighbouring double -- no implementation can then agree with
    every libm (glibc's exp is wrong by one unit in ~1 % of the last places; its FMA and non-FMA variants differ too)."""
    import math
    return (U < math.exp(lp)) == (U < _exp_correctly_rounded(lp))     # math.exp: the C library's, like numba's and the oracle's


def test_device_exp_is_correctly_rounded():
    """rx_exp_cr (the tie-break's exp, double-double) against 60-digit arithmetic: random arguments over the range the
    mixing kernels can meet, and the worst case for the decision: x = log(U), where exp(x) is within an ulp of U."""
    rng = np.random.default_rng(11)
    U = (rng.integers(1, 2 ** 53, 1500).astype(np.float64)) / 2.0 ** 53
    x = np.concatenate([-40.0 * rng.random(1500), np.log(U), rng.uniform(-745.0, 709.0, 300),
                        [0.0, -0.0, 1.0, -1.0, 709.78, -745.13, -745.14, -800.0, 710.0, -1e-300, 1e-17, -36.7368005696771]])
    e = gpu_engine(0, 2, 2)
    y = e.selftest_exp(x)
    e.close()
    with np.errstate(over='ignore'):
        ref = np.array([_exp_correctly_rounded(v) if v < 709.79 else np.inf for v in x])
    bad = np.flatnonzero(y != ref)
    assert bad.size == 0, [(x[b], y[b], ref[b]) for b in bad[:5]]
    # (for the record: how often the host libm itself is not correctly rounded on the same arguments)
    import math
    libm = np.array([math.exp(v) if v < 709.78 else np.inf for v in x])
    print('libm exp differs from the correctly rounded value at %d of %d arguments' % (int(np.sum(libm != ref)), x.size))


def test_swap_all_tie_break_inside_the_guard_band_any_k():
    """The same for K = 3 (k_mix_walk2c: rejection-sampled indices, the exact decision of w2c_exact_decision)."""
    from oracle import oracle
    hits = 0; undecidable = 0
    for seed in range(40):
        mt = oracle.MT(seed)
        while True:
            i, j = mt.randint(3), mt.randint(3)
            if i != j: break
        U = mt.rand()
        for rel in (0.0, 1e-14, -1e-14, 1e-12, -1e-12, 1e-10, -1e-10):
            lp = np.log(U) * (1.0 + rel)
            if not _libm_decides_like_exact_arithmetic(U, lp): undecidable += 1; continue
            u = np.zeros((3, 3)); u[i, j] = u[j, i] = -0.5 * lp      # log_p(i, j) = lp under the identity permutation
            e = gpu_engine(0, 3, 3)
            e.set_energies(u); e.set_replica_states(np.arange(3)); e.mix_seed(seed, 0)
            st, nacc, nprop = e.mix_swap_all(6000)
            stats = e.mix_stats()
            hits += stats['exact_exp'] > 0
            assert stats['rounds'] > 0
            e.close()
            mo = oracle.MT(seed); st_o = np.arange(3, dtype=np.int64)
            na = np.zeros((3, 3), np.int64); npr = np.zeros((3, 3), np.int64)
            oracle.mix_swap_all(mo, 6000, st_o, u, na, npr)
            assert np.array_equal(st, st_o) and np.array_equal(nacc, na) and np.array_equal(nprop, npr), (seed, rel)
    assert hits > 100   # the exact path really ran
    assert undecidable <= 6   # (cases where the host libm's exp is itself off by one in the last place and that decides)


@pytest.mark.parametrize('nswap', [40, 6000])
def test_swap_all_tie_break_inside_the_guard_band(nswap):
    """The one place where the decision is not taken in the log domain: |log_p - log U| <= 1e-9, where the kernels fall back to
    the reference's own test U < exp(log_p).  K = 2 matrices are built so that the first attempt with i != j lands inside
    the band (log_p = log U to a relative 0, 1e-14, 1e-12, 1e-10 on either side), for 60 seeds; nswap = 40 runs in the
    pass-tail kernel (k_mix_walk_pow2), 6000 in k_mix_walk2."""
    from oracle import oracle
    hits = 0; undecidable = 0
    for seed in range(60):
        mt = oracle.MT(seed)
        while True:
            i, j = mt.randint(2), mt.randint(2)
            if i != j: break
        U = mt.rand()
        for rel in (0.0, 1e-14, -1e-14, 1e-12, -1e-12, 1e-10, -1e-10):
            lp = np.log(U) * (1.0 + rel)
            if not _libm_decides_like_exact_arithmetic(U, lp): undecidable += 1; continue
            u = np.array([[0.0, -0.5 * lp], [-0.5 * lp, 0.0]])      # log_p(0, 1) = -(u01 + u10) + u00 + u11 = lp
            e = gpu_engine(0, 2, 2)
            e.set_energies(u); e.set_replica_states(np.arange(2)); e.mix_seed(seed, 0)
            st, nacc, nprop = e.mix_swap_all(nswap)
            hits += e.mix_stats()['exact_exp'] > 0
            e.close()
            mo = oracle.MT(seed); st_o = np.arange(2, dtype=np.int64)
            na = np.zeros((2, 2), np.int64); npr = np.zeros((2, 2), np.int64)
            oracle.mix_swap_all(mo, nswap, st_o, u, na, npr)
            assert np.array_equal(st, st_o) and np.array_equal(nacc, na) and np.array_equal(nprop, npr), (seed, rel)
    assert hits > 100   # the exact path really ran
    assert undecidable <= 8


def test_unseeded_stream_is_an_error():
    from openmmtools_b200._engine import EngineError
    e = gpu_engine(0, 4, 4)
    with pytest.raises(EngineError):
        e.mix_swap_all(10)
    e.close()


@pytest.mark.parametrize('K', [16, 64, 256])
def test_swap_all_with_nonfinite_and_huge_energies(K):
    """NaN, +/-inf and 1e300 entries (a decoupled atom on top of another one gives astronomically large energies):
    the reference's IEEE semantics (NaN compares false, exp(-inf) = 0) must be reproduced exactly, also through the
    K=256 row-image filter (which must fall back to the exact path)."""
    from oracle import oracle
    u = energies('flat', K, 31337 + K)
    rng = np.random.default_rng(K)
    for v in (np.nan, np.inf, -np.inf, 1e300, -1e300, 2.4e6):
        for _ in range(max(2, K // 16)):
            u[rng.integers(K), rng.integers(K)] = v
    for variant in range(2):
        if variant == 1:
            u = np.where(np.isfinite(u) & (np.abs(u) < 1e7), u, 1e6)   # finite, huge dynamic range per row: filter path
        e = gpu_engine(0, K, K)
        e.set_energies(u)
        e.set_replica_states(np.arange(K))
        e.mix_seed(99, 0)
        mt = oracle.MT(99)
        st_o = np.arange(K, dtype=np.int64)
        nswap = min(K ** 3, 2_000_000)
        for it in range(2):
            st, nacc, nprop = e.mix_swap_all(nswap)
            na = np.zeros((K, K), np.int64); npr = np.zeros((K, K), np.int64)
            oracle.mix_swap_all(mt, nswap, st_o, u, na, npr)
            assert np.array_equal(st, st_o), (K, variant, it)
            assert np.array_equal(nacc, na) and np.array_equal(nprop, npr)
        e.close()


@pytest.mark.parametrize('K,model', [(16, 'flat'), (64, 'normal'), (128, 'flat'), (256, 'flat'), (1024, 'flat')])
def test_swap_all_pow2_walkers_vs_oracle(K, model):
    """Both power-of-two walkers at up to 1.5 M attempts per call: the row-image filter (k_mix_walk2 and k_mix_walk_pow2<true>,
    K <= 256) and the exact values from L2 every round (k_mix_walk_pow2<false>, K >= 512)."""
    from oracle import oracle
    u = energies(model, K, 977 + K)
    e = gpu_engine(0, K, K)
    e.set_energies(u)
    e.set_replica_states(np.arange(K))
    e.mix_seed(21, 0)
    mt = oracle.MT(21)
    st_o = np.arange(K, dtype=np.int64)
    nswap = min(K ** 3, 1_500_000)
    for it in range(2):
        st, nacc, nprop = e.mix_swap_all(nswap)
        na = np.zeros((K, K), np.int64); npr = np.zeros((K, K), np.int64)
        oracle.mix_swap_all(mt, nswap, st_o, u, na, npr)
        assert np.array_equal(st, st_o), (K, it)
        assert np.array_equal(nacc, na) and np.array_equal(nprop, npr)
    e.close()
