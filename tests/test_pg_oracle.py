"""Moment checks of the CPU Polya-Gamma restatement (oracle/pg.py)."""
import numpy as np
import pytest
from oracle import pg


@pytest.mark.parametrize('b', [1, 3, 2.5, 0.4, 250.0])
@pytest.mark.parametrize('z', [0.0, 1.0, 4.0])
def test_pg_moments(b, z):
    rng = np.random.default_rng(int(b * 10 + z))
    n = 30000
    x = pg.pgdraw(np.full(n, float(b)), np.full(n, z), rng)
    m, v = float(pg.pg_mean(b, z)), float(pg.pg_var(b, z))
    assert abs(x.mean() - m) < 5 * np.sqrt(v / n)
    assert abs(x.var() / v - 1) < 0.08


def test_pg_zero_for_missing():
    rng = np.random.default_rng(0)
    x = pg.pgdraw(np.array([np.nan, 0.0, -2.0]), np.array([0.3, 0.3, 0.3]), rng)
    assert np.all(x == 0)


def _pg_var_mp(z):
    """Var PG(1, z) = (sinh z - z) / (4 z^3 cosh^2(z/2)) in 60-digit arithmetic (no overflow there)."""
    import mpmath
    with mpmath.workdps(60):
        z = mpmath.mpf(z)
        return float((mpmath.sinh(z) - z) / (4 * z ** 3 * mpmath.cosh(z / 2) ** 2))


@pytest.mark.parametrize('z', [2e-3, 0.1, 1.0, 12.0, 100.0, 700.0, 712.0, 1000.0, 1e4, -300.0])
def test_pg_var_closed_form(z):
    """The closed form stays finite and exact past z = 710, where sinh and cosh^2 overflow; (sinh z - z) cancels to
    ~eps / z^2 relative for small z, hence the looser bound at z = 2e-3."""
    want = _pg_var_mp(abs(z))
    got = float(pg.pg_var(1.0, z))
    assert np.isfinite(got) and abs(got / want - 1) < (1e-9 if abs(z) < 0.01 else 1e-13), (got, want)
    assert float(pg.pg_var(200.0, z)) == pytest.approx(200.0 * got, rel=1e-15)


def test_pg_tail_mass_at_large_z():
    """P(exponential tail) of the Devroye proposal: finite in (0, 1), then exactly 0 where q/p would overflow (|z| > ~97)."""
    Z = np.array([0.0, 1.0, 10.0, 40.0, 150.0, 500.0])
    with np.errstate(over='raise', invalid='raise', divide='raise'):
        p = pg._mass_texpon(Z)
    assert np.all((p[:4] > 0) & (p[:4] < 1)) and np.all(p[4:] == 0.0)
    assert np.all(np.diff(p) <= 0)


@pytest.mark.parametrize('b', [1, 2.5, 250.0])
@pytest.mark.parametrize('z', [30.0, -100.0, 300.0, 1000.0])
def test_pg_moments_large_z(b, z):
    """Large tilts (Binomial cells with near-certain outcomes): the reference the device sampler is tested against
    must itself be right there - the exact sampler past the q/p overflow, the normal route past z = 710."""
    rng = np.random.default_rng(int(b * 10) + int(abs(z)))
    n = 30000
    x = pg.pgdraw(np.full(n, float(b)), np.full(n, z), rng)
    m, v = float(pg.pg_mean(b, z)), float(pg.pg_var(b, z))
    assert np.all(x > 0)
    assert abs(x.mean() - m) < 5 * np.sqrt(v / n)
    assert abs(x.var() / v - 1) < 0.08
