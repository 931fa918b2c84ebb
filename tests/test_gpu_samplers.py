"""Moment / distribution checks of the on-device Philox samplers (no reference source
exists for pypolyagamma offline, so PG parity is by moments: SURVEY.md 8c)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _z(sample, mean, var):
    return (sample.mean() - mean) / np.sqrt(var / sample.size)


def test_normal_uniform_exponential_moments():
    from functionalmf_b200.engine import rng_sample
    from scipy import stats
    n = 400000
    x = rng_sample('normal', n, seed=11)
    assert abs(_z(x, 0.0, 1.0)) < 5 and abs(x.var() - 1.0) < 0.02
    assert stats.kstest(x[:100000], 'norm').pvalue > 1e-4
    u = rng_sample('uniform', n, seed=12)
    assert u.min() > 0.0 and u.max() < 1.0
    assert stats.kstest(u[:100000], 'uniform').pvalue > 1e-4
    e = rng_sample('exponential', n, seed=13)
    assert abs(_z(e, 1.0, 1.0)) < 5


@pytest.mark.parametrize('shape', [0.1, 0.5, 1.0, 2.5, 8.5, 1000.0])
def test_gamma_moments(shape):
    from functionalmf_b200.engine import rng_sample
    from scipy import stats
    g = rng_sample('gamma', 300000, param=shape, seed=int(shape * 10) + 1)
    assert np.all(g >= 0)
    assert abs(_z(g, shape, shape)) < 5
    assert abs(g.var() / shape - 1.0) < 0.05
    if shape >= 0.5:
        assert stats.kstest(g[:50000], 'gamma', args=(shape,)).pvalue > 1e-4


@pytest.mark.parametrize('b', [1.0, 2.0, 4.0, 2.5, 0.3, 30.0, 200.0])
@pytest.mark.parametrize('z', [0.0, 0.5, 2.0, 5.0, -12.0, 30.0, -100.0, 300.0, 1000.0])
def test_polya_gamma_moments(b, z):
    # |z| >= 100: past the overflow of q/p in the Devroye set-up (exact sampler) and, with b = 200, past z = 710
    # where the closed-form variance of the normal route is inf / inf
    from functionalmf_b200.engine import pg_sample
    from oracle import pg as OPG
    n = 60000 if b <= 4 else 20000
    x = pg_sample(np.full(n, b), np.full(n, z), seed=int(10 * b) + int(abs(z)) + 1)
    m, v = float(OPG.pg_mean(b, z)), float(OPG.pg_var(b, z))
    assert np.all(x > 0)
    assert abs(_z(x, m, v)) < 5, (x.mean(), m)
    assert abs(x.var() / v - 1.0) < 0.08, (x.var(), v)


def test_polya_gamma_matches_cpu_oracle_distribution():
    """Two-sample KS between the device sampler and the CPU restatement."""
    from functionalmf_b200.engine import pg_sample
    from oracle import pg as OPG
    from scipy import stats
    rng = np.random.default_rng(3)
    for b, z in [(1.0, 0.0), (1.0, 3.0), (4.0, 1.0), (2.5, 1.0), (1.0, 100.0), (2.5, -150.0)]:
        n = 40000
        gpu = pg_sample(np.full(n, b), np.full(n, z), seed=77)
        cpu = OPG.pgdraw(np.full(n, b), np.full(n, z), rng)
        assert stats.ks_2samp(gpu, cpu).pvalue > 1e-4, (b, z)


def test_pg_missing_cells_are_zero():
    from functionalmf_b200.engine import pg_sample
    x = pg_sample(np.array([0.0, np.nan, -1.0, 3.0]), np.array([1.0, 1.0, 1.0, np.nan]))
    assert np.all(x == 0.0)
