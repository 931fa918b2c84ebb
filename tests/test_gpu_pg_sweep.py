"""omega as a sweep draws it: the Polya-Gamma step of a Binomial / negative-binomial engine, on every route of
launch_pg_draw (pg_kernels.cu), against the closed-form moments and the CPU sampler of oracle/pg.py.

tests/test_gpu_samplers.py checks pg_draw() through a flat one-thread-per-value kernel.  The sweep reaches it through
kernels with their own indexing, psi = w.v computation, trial-count prefetch and lane splitting:
  * pg_draw_group_kernel<G = 8 | 4 | 2>: G lanes per cell (each with its own Philox stream) while cells * 2G <= 2^20;
  * pg_draw_kernel<KMAX = 8 | 16 | 32>: one thread per cell, W staged in shared memory per 32-row block, the
    observed flag and trial count of the next row loaded while the current row is sampled.
With the sample mask set to the nu2 bit alone a sweep only draws omega, so W and V stay as set and psi = W V^T is
known on the host.  Every draw is standardised with the exact mean and variance of PG(b, psi); the standardised
values must have mean 0 and second moment 1 overall and in buckets where an indexing or prefetch slip would show
(row mod 32, the last partial row block, the last partial column tile, each trial count, each sampler regime of
|psi|).  A second design with one (b, psi) per bucket compares the whole law with oracle/pg.py (two-sample KS).
"""
import numpy as np
import pytest

from functionalmf_b200._lib import BINOMIAL, NEGBINOMIAL, SAMPLE_NU2

pytestmark = pytest.mark.gpu

# trial counts: integers, fractional values (floor(b) exact draws + the sum-of-gammas series), and b > 170 (normal)
B_VALUES = [1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 7.0, 8.0, 0.3, 2.5, 7.75, 200.0, 1000.0]
# sampler regimes of |psi| (Z = |psi| / 2): 0; Z <= 1/t (truncated-Levy inverse-Gaussian proposal); Z < 12 (direct
# set-up); Z >= 12 (log-space set-up); |psi| > 97 (q/p past the floating-point range)
PSI_EDGES = [0.0, 3.125, 24.0, 97.0]

# (route, N, M, T, K): the per-cell shapes have N = 300 (not a multiple of 32) and P = 2000 (not a multiple of 256)
ROUTES = [
    ('group8', 64, 32, 32, 3),
    ('group4', 100, 40, 50, 5),
    ('group2', 150, 50, 50, 7),
    ('cell8', 300, 40, 50, 5),
    ('cell16', 300, 40, 50, 12),
    ('cell32', 300, 40, 50, 32),
]


def pg_route(cells, K):
    """The kernel launch_pg_draw picks, restated: lane groups of G = 2, 4, 8 while cells * 2G <= 2^20, else one
    thread per cell with KMAX = 8 / 16 / 32."""
    G = 1
    while G < 8 and cells * 2 * G <= (1 << 20):
        G *= 2
    if G > 1:
        return 'group%d' % G
    return 'cell%d' % (8 if K <= 8 else 16 if K <= 16 else 32)


def _binomial_engine(N, M, T, K, Nt, W, V, seed=21):
    from functionalmf_b200.engine import Engine
    eng = Engine(N, M, T, nembeds=K, tf_order=2, likelihood=BINOMIAL, seed=seed, use_graph=0)
    Ys = np.where(np.isnan(Nt), np.nan, np.floor(np.nan_to_num(Nt) / 2))
    eng.set_data_binomial(Ys.reshape(N, M, T), Nt.reshape(N, M, T))
    eng.set('W', W)
    eng.set('V', V)
    eng.set_sample_mask(SAMPLE_NU2)
    return eng


def _standardise(omega, b, psi):
    from oracle import pg as OPG
    return (omega - OPG.pg_mean(b, psi)) / np.sqrt(OPG.pg_var(b, psi))


def _check_moments(u, label, min_n=500):
    """mean u = 0 and mean u^2 = 1 within 5 standard errors, each taken from the sample's own moments."""
    n = u.size
    assert n >= min_n, (label, n)
    m1, m2 = u.mean(), (u * u).mean()
    se1, se2 = u.std() / np.sqrt(n), (u * u).std() / np.sqrt(n)
    assert abs(m1) < 5 * se1, (label, n, m1, se1)
    assert abs(m2 - 1.0) < 5 * se2, (label, n, m2, se2)


def _mixed_design(rs, N, P, K):
    cls = rs.random_sample((N, P))
    b = np.where(cls < 0.6, rs.randint(1, 9, size=(N, P)).astype(float),
                 np.where(cls < 0.85, rs.choice([0.3, 2.5, 7.75], size=(N, P)), rs.choice([200.0, 1000.0], size=(N, P))))
    b[rs.random_sample((N, P)) < 0.1] = np.nan
    # psi = a_i c_p + (a small row-dependent part): c_p from the five regimes, the part left out where c_p = 0
    reg = rs.randint(0, 5, size=P)
    lo = np.array([0.0, 0.0, 2.0, 15.0, 60.0])[reg]
    hi = np.array([0.0, 2.0, 15.0, 60.0, 500.0])[reg]
    c = rs.uniform(lo, hi) * rs.choice([-1.0, 1.0], size=P)
    W = np.empty((N, K))
    W[:, 0] = rs.uniform(0.6, 1.6, size=N) * rs.choice([-1.0, 1.0], size=N)
    W[:, 1:] = 0.3 * rs.normal(size=(N, K - 1))
    V = np.zeros((P, K))
    V[:, 0] = c
    V[:, 1:] = 0.3 * rs.normal(size=(P, K - 1)) * (reg != 0)[:, None]
    return b, W, V


@pytest.mark.parametrize('route,N,M,T,K', ROUTES)
def test_sweep_omega_standardised_moments(route, N, M, T, K):
    P = M * T
    assert pg_route(N * P, K) == route
    rs = np.random.RandomState(N + 7 * K)
    b, W, V = _mixed_design(rs, N, P, K)
    psi = W @ V.T
    obs = ~np.isnan(b)
    eng = _binomial_engine(N, M, T, K, b, W, V)
    eng.sweep(1)
    om = eng.get('omega').reshape(N, P)
    assert np.all(om[~obs] == 0.0)
    assert np.all(np.isfinite(om[obs])) and np.all(om[obs] > 0.0)
    u = np.zeros((N, P))
    u[obs] = _standardise(om[obs], b[obs], psi[obs])
    _check_moments(u[obs], 'all')
    rows = np.arange(N)[:, None] + np.zeros((1, P), dtype=int)
    cols = np.zeros((N, 1), dtype=int) + np.arange(P)[None, :]
    for r in range(32):
        _check_moments(u[obs & (rows % 32 == r)], ('row mod 32', r))
    _check_moments(u[obs & (rows >= (N - 1) // 32 * 32)], 'last row block')
    _check_moments(u[obs & (cols >= (P - 1) // 256 * 256)], 'last column tile')
    for bv in B_VALUES:
        _check_moments(u[obs & (b == bv)], ('b', bv), min_n=300)
    apsi = np.abs(psi)
    pcls = np.where(apsi == 0.0, 0, 1 + np.searchsorted(PSI_EDGES[1:], apsi, side='right'))
    for k in range(5):
        _check_moments(u[obs & (pcls == k)], ('|psi| class', k))

    # repeatability: the same seed gives the same bits; the next sweep gives new, uncorrelated draws
    twin = _binomial_engine(N, M, T, K, b, W, V)
    twin.sweep(1)
    assert np.array_equal(twin.get('omega').reshape(N, P), om)
    twin.close()
    eng.sweep(1)
    om2 = eng.get('omega').reshape(N, P)
    assert np.all(om2[~obs] == 0.0)
    assert not np.any(om2[obs] == om[obs])
    u2 = _standardise(om2[obs], b[obs], psi[obs])
    _check_moments(u2, 'second sweep')
    n = u2.size
    assert abs(np.corrcoef(u[obs], u2)[0, 1]) < 5 / np.sqrt(n)
    eng.close()


# (b, psi) pairs of the exact-law comparison: row group g has b = PAIRS[g][0], column group g has psi = PAIRS[g][1]
PAIRS = [(1.0, 0.0), (2.5, 3.0), (4.0, 100.0), (7.75, -30.0)]


@pytest.mark.parametrize('route,N,M,T,K', ROUTES)
def test_sweep_omega_law_matches_cpu_sampler(route, N, M, T, K):
    from oracle import pg as OPG
    from scipy import stats
    P = M * T
    assert pg_route(N * P, K) == route
    G = len(PAIRS)
    rg, cg = np.arange(N) * G // N, np.arange(P) * G // P
    b = np.repeat(np.array([p[0] for p in PAIRS])[rg][:, None], P, axis=1)
    W = np.zeros((N, K))
    W[:, 0] = 1.0
    V = np.zeros((P, K))
    V[:, 0] = np.array([p[1] for p in PAIRS])[cg]
    eng = _binomial_engine(N, M, T, K, b, W, V, seed=5)
    smallest = min(np.sum(rg == g) * np.sum(cg == g) for g in range(G))
    nsw = -(-20000 // smallest)
    draws = [[] for _ in range(G)]
    for _ in range(nsw):
        eng.sweep(1)
        om = eng.get('omega').reshape(N, P)
        for g in range(G):
            draws[g].append(om[np.ix_(rg == g, cg == g)].ravel())
    eng.close()
    rng = np.random.default_rng(N + K)
    for g, (bv, zv) in enumerate(PAIRS):
        x = np.concatenate(draws[g])
        assert x.size >= 20000
        ref = OPG.pgdraw(np.full(x.size, bv), np.full(x.size, zv), rng)
        p = stats.ks_2samp(x, ref).pvalue
        assert p > 1e-4, (route, bv, zv, p)


def test_negbin_pseudo_counts_and_omega():
    """Negative binomial: the PG step draws PG(sum_obs (y + R), psi) with kappa = sum_obs y - N/2.  A per-cell,
    fractional R makes every trial count fractional; counts of up to a few hundred put part of them on the normal
    route (b > 170)."""
    from oracle import btf_oracle as O
    from functionalmf_b200.engine import Engine
    N, M, T, R, K = 150, 20, 40, 2, 6
    P = M * T
    rs = np.random.RandomState(3)
    W = rs.normal(size=(N, K)) * 0.8
    V = rs.normal(size=(M, T, K)) * 0.8
    Mu = np.einsum('nk,mtk->nmt', W, V)
    lam = rs.gamma(5.0, np.exp(np.clip(Mu, -4.0, 3.5)))[..., None] * np.ones(R)
    Y = rs.poisson(lam).astype(float)
    Y[rs.random_sample(Y.shape) < 0.3] = np.nan
    Rd = rs.uniform(0.5, 20.0, size=(N, M, T))
    eng = Engine(N, M, T, nembeds=K, tf_order=2, likelihood=NEGBINOMIAL, seed=13, use_graph=0, rdims_mask=0)
    eng.set_data_negbin(Y)
    eng.set('W', W)
    eng.set('V', V)
    eng.set('R', Rd)
    eng.set_sample_mask(SAMPLE_NU2)
    eng.sweep(1)
    _, Nref = O.step_R(Rd, W, V, Y, [], np.zeros((0, N, M, T)), np.zeros((0, N, M, T)))
    obs = np.any(~np.isnan(Y), axis=-1)
    assert np.all(np.asarray(eng.get('R')) == Rd)
    Ng, kap = eng.get('Ntrials'), eng.get('kappa')
    assert np.max(np.abs(Ng[obs] / Nref[obs] - 1.0)) < 1e-12
    assert np.all(Ng[~obs] == 0.0) and np.all(kap[~obs] == 0.0)
    kref = np.nansum(Y, axis=-1) - Nref / 2
    assert np.max(np.abs(kap[obs] - kref[obs]) / np.abs(Nref[obs])) < 1e-12
    assert np.sum(Nref[obs] > 170) > 2000 and np.sum(Nref[obs] < 170) > 2000
    om = eng.get('omega')
    assert np.all(om[~obs] == 0.0) and np.all(np.isfinite(om[obs])) and np.all(om[obs] > 0.0)
    psi = Mu
    u = _standardise(om[obs], Nref[obs], psi[obs])
    _check_moments(u, 'negbin all')
    _check_moments(u[Nref[obs] > 170], 'negbin b > 170')
    _check_moments(u[Nref[obs] < 170], 'negbin b < 170')
    eng.close()
