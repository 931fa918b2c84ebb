"""Constrained model with the built-in Gaussian likelihood (loglikelihood='gaussian', data Y [N, M, T(, R)], mean
W V^T, noise variance nu2 sampled, fixed, or known per cell): the GASS steps run inside the engine's sweep
(gass_kernels.cu).  Every random choice of a transition is a function of ngrid + 2 injected uniforms per row / column,
so the device steps are compared exactly with the host gass() driven by the same uniforms and a numpy Gaussian
callable."""
import os
import warnings
import numpy as np
import pytest
from scipy.stats import norm

from test_gpu_constrained_poisson import UniformRng, _device_step

pytestmark = pytest.mark.gpu


class GaussianLL(object):
    """nansum(scipy.stats.norm.logpdf(Y, W V^T, sqrt(nu2))) over a row or a column of cells; nu2 is a scalar or an
    [N, M, T] array, and a cell whose variance is +inf counts as missing."""

    def __init__(self, nu2):
        self.nu2 = nu2

    def __call__(self, Y, WV, W, V, row=None, col=None):
        nu2 = np.broadcast_to(np.asarray(self.nu2, dtype=float), Y.shape[:3])
        if row is not None:
            Y, nu2 = Y[row], nu2[row]
        if col is not None:
            Y, nu2 = Y[:, col], nu2[:, col]
        if Y.ndim > WV.ndim:
            WV, nu2 = WV[..., None], nu2[..., None]
        Y = np.where(np.isinf(nu2), np.nan, Y)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore', category=RuntimeWarning)
            return np.nansum(norm.logpdf(Y, WV, np.sqrt(nu2)))


def box(T, lo, hi):
    """lo <= Mu <= hi in every cell."""
    return np.concatenate([np.concatenate([np.eye(T), -np.eye(T)]), np.concatenate([np.full(T, lo), np.full(T, -hi)])[:, None]],
                          axis=1)


def monotone(T):
    """Mu[i, j, t + 1] >= Mu[i, j, t]."""
    A = np.zeros((T - 1, T))
    A[np.arange(T - 1), np.arange(T - 1)] = -1.0
    A[np.arange(T - 1), np.arange(1, T)] = 1.0
    return np.concatenate([A, np.zeros((T - 1, 1))], axis=1)


# ------------------------------------------------------------------ 1. the host gass() with the same uniforms
def _case(kind, rs):
    N, M, T, K, R = 7, 4, 8, 3, 3
    W = rs.uniform(0.1, 1.5, size=(N, K))
    W[np.triu_indices(K, k=1)] = 0
    V = (rs.uniform(0.0, 0.3, size=(M, T, K))).cumsum(axis=1)       # non-decreasing in t: Mu is, since W >= 0
    nu2 = 0.3
    kw = {}
    if kind == 'offset':
        # |y| ~ 1e4 with noise ~ 1: the expanded square sum y^2 - 2 tau sum y + n tau^2 would lose the value
        W[:, 0] = 100.0 + rs.uniform(size=N)
        V[:, :, 0] += 100.0
        nu2 = 1.0
    if kind in ('percell', 'percell_ep'):
        nu2 = rs.uniform(0.1, 0.6, size=(N, M, T))
        nu2[rs.random_sample(nu2.shape) < 0.1] = np.inf
    if kind == 'coarse':
        W = rs.normal(size=(N, K)); W[np.triu_indices(K, k=1)] = 0
        V = rs.normal(size=(M, T, K))
    Mu = np.einsum('nk,mtk->nmt', W, V)
    sd = np.sqrt(np.where(np.isinf(nu2), 1.0, nu2)) * np.ones((N, M, T))
    Y = Mu[..., None] + sd[..., None] * rs.normal(size=(N, M, T, R))
    Y[rs.random_sample(Y.shape) < 0.2] = np.nan
    Y[3] = np.nan                                          # an all-missing row
    if kind == '3d':
        Y = Y[..., 0]
    cons = box(T, Mu.min() - 0.5 if kind == 'offset' else 0.0, Mu.max() + 1.0)
    if kind == 'monotone':
        cons = monotone(T)
    if kind == 'coarse':
        cons = box(T, -1e8, 1e8)                           # no constraint is ever active: the coarse grid
    if kind == 'rowcons':
        kw['Row_constraints'] = np.array([[1.0, 0.0, 0.0, 0.05], [0.0, -1.0, -1.0, -5.0]])     # w_0 >= 0.05, w_1 + w_2 <= 5
    if kind in ('ep', 'percell_ep'):
        kw['ep_approx'] = (Mu + 0.1 * rs.normal(size=Mu.shape), 0.2 + 0.3 * rs.random_sample(Mu.shape))
    if kind == 'offset':
        kw['ep_approx'] = (Mu + 0.1 * rs.normal(size=Mu.shape), np.ones(Mu.shape))
    return N, M, T, K, W, V, Y, nu2, cons, kw


CASES = [('box', 10), ('box', 40), ('box', 100), ('monotone', 10), ('monotone', 40), ('monotone', 100), ('rowcons', 40),
         ('ep', 10), ('ep', 100), ('coarse', 40), ('3d', 40), ('offset', 40), ('percell', 40), ('percell_ep', 40),
         ('slice', 40)]


@pytest.mark.parametrize('kind,ngrid', CASES)
def test_device_gass_matches_host_gass(kind, ngrid, monkeypatch):
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    from functionalmf_b200 import constrained, gass as G
    rs = np.random.RandomState(31 + ngrid + len(kind))
    N, M, T, K, W, V, Y, nu2, cons, kw = _case(kind, rs)
    common = dict(nembeds=K, tf_order=1, gass_ngrid=ngrid, sigma2_init=1.0, lam2_init=0.5, W_init=W, V_init=V, seed=5,
                  **kw)
    host = CM(N, M, T, GaussianLL(nu2), cons, **common)
    dev = CM(N, M, T, 'gaussian', cons, nu2_true=nu2, **common)
    log = []

    def recording_gass(x, v, ll, Cons, mu=None, ll_args=None, ngrid=100, rng=None):
        mu_ = np.zeros_like(x) if mu is None else mu
        A, c = Cons[:, :-1], Cons[:, -1]
        log.append(len(G.feasible_angles(A.dot(x - mu_), A.dot(v), c - A.dot(mu_), ngrid)))
        return G.gass(x, v, ll, Cons, mu=mu, ll_args=ll_args, ngrid=ngrid, rng=rng)
    monkeypatch.setattr(constrained, 'gass', recording_gass)

    for which in ('W', 'V'):
        n = N if which == 'W' else M
        U = rs.random_sample((n, ngrid + 2))
        if kind == 'slice':
            U[:, 0] = 1.0 - 1e-16          # height = current ll: often no candidate clears it
        zz = rs.normal(size=(N, K) if which == 'W' else (M, T, K))
        del log[:]
        host.W, host.V = W.copy(), V.copy()
        host._rng = UniformRng(U)
        host._sync_ep()
        if which == 'W':
            host._resample_W(Y, z=zz)
        else:
            host._resample_V(Y, z=zz)
        new, d = _device_step(dev, Y, which, U, zz, W=W, V=V)
        ref = host.W if which == 'W' else host.V
        assert np.array_equal(d[:, 0].astype(int), np.array(log)), (d[:, 0], log)
        assert np.allclose(new, ref, rtol=1e-9, atol=1e-9), np.abs(new - ref).max()
        if kind == 'coarse':
            assert np.all(d[:, 0] == ngrid)
        if kind == 'slice':
            assert np.any(d[:, 1] == 0) or np.any(d[:, 1] < np.minimum(d[:, 0], ngrid))
        if which == 'W':
            assert np.all(new[np.triu_indices(K, k=1)] == 0)
        if kind in ('box', 'monotone', 'rowcons', 'ep', 'offset', 'percell', 'percell_ep'):
            assert np.any(d[:, 1] > 0) and not np.array_equal(new, W if which == 'W' else V)


# ------------------------------------------------------------------ 2. the nu2 step
def _chain_model(seed=11, R=2, **kw):
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    rs = np.random.RandomState(4)
    N, M, T, K = 9, 5, 12, 3
    W = rs.uniform(0.2, 0.8, size=(N, K)); W[np.triu_indices(K, k=1)] = 0
    V = rs.uniform(0.0, 0.3, size=(M, T, K)).cumsum(axis=1)
    Mu = np.einsum('nk,mtk->nmt', W, V)
    Y = Mu[..., None] + 0.3 * rs.normal(size=(N, M, T, R))
    Y[rs.random_sample(Y.shape) < 0.1] = np.nan
    m = CM(N, M, T, 'gaussian', monotone(T), nembeds=K, tf_order=1, gass_ngrid=40, W_init=W, V_init=V, seed=seed, **kw)
    return m, Y


def test_nu2_step_uses_the_current_residual():
    m, Y = _chain_model(nu2_a=0.7, nu2_b=0.4)
    assert m.sample_nu2
    for _ in range(3):
        W, V = m.W.copy(), m.V.copy()
        m.resample(Y)
        resid = np.nansum((Y - np.einsum('nk,mtk->nmt', W, V)[..., None]) ** 2)
        a, b, n_obs = m._engine.diag('nu2_rate')
        assert n_obs == np.sum(~np.isnan(Y))
        assert abs(a - (0.7 + n_obs / 2)) <= 1e-10 * a
        assert abs(b - (0.4 + resid / 2)) <= 1e-10 * b, (b, 0.4 + resid / 2)


# ------------------------------------------------------------------ 3. chains
def test_chain_keeps_constraints_and_is_reproducible():
    m1, Y = _chain_model()
    r1 = m1.run_gibbs(Y, nburn=5, nthin=2, nsamples=6, verbose=False)
    Mu = np.einsum('znk,zmtk->znmt', r1['W'], r1['V'])
    assert np.all(np.diff(Mu, axis=-1) >= -1e-9)
    assert not np.array_equal(r1['W'][0], r1['W'][-1])
    assert r1['nu2'].shape == (6, 1) and len(np.unique(r1['nu2'])) == 6
    m2, _ = _chain_model()
    r2 = m2.run_gibbs(Y, nburn=5, nthin=2, nsamples=6, verbose=False)
    for k in ('W', 'V', 'Tau2', 'sigma2', 'lam2', 'nu2'):
        assert np.array_equal(r1[k], r2[k]), k
    # the per-sweep loop (eager engine, one btf_sweep per resample) against run_gibbs (graph replay in segments)
    m3, _ = _chain_model(use_graph=0)
    S = []
    for step in range(5 + 2 * 6):
        m3.resample(Y)
        if step >= 5 and (step - 5) % 2 == 0:
            S.append((m3.W.copy(), m3.V.copy(), float(m3.nu2)))
    assert np.array_equal(np.array([s[0] for s in S]), r1['W'])
    assert np.array_equal(np.array([s[1] for s in S]), r1['V'])
    assert np.array_equal(np.array([s[2] for s in S]), r1['nu2'][:, 0])


def _variances(rs, inf_frac=0.1):
    """known variances of the chain model's cells, some of them +inf"""
    nu2 = rs.uniform(0.05, 0.2, size=(9, 5, 12))
    nu2[rs.random_sample(nu2.shape) < inf_frac] = np.inf
    return nu2


@pytest.mark.parametrize('mode', ['scalar', 'percell'])
def test_checkpoint_resumes_bit_for_bit(tmp_path, mode):
    kw = {} if mode == 'scalar' else {'nu2_true': _variances(np.random.RandomState(2))}
    m, Y = _chain_model(**kw)
    for _ in range(3):
        m.resample(Y)
    path = str(tmp_path / 'ck.npz')
    m.save_checkpoint(path)
    if mode == 'scalar':
        assert 'nu2' in np.load(path).files
    ra = m.run_gibbs(Y, nburn=2, nthin=1, nsamples=3, verbose=False)
    m2, _ = _chain_model(**kw)
    m2._upload(Y)
    m2.load_checkpoint(path)
    rb = m2.run_gibbs(Y, nburn=2, nthin=1, nsamples=3, verbose=False)
    for k in ('W', 'V', 'nu2'):
        assert np.array_equal(ra[k], rb[k]), k
    if mode == 'percell':
        nu2 = kw['nu2_true']
        assert ra['nu2'].shape == (3,) + nu2.shape and not ra['nu2'].flags.writeable
        assert np.array_equal(ra['nu2'], np.broadcast_to(nu2, ra['nu2'].shape))


def test_track_mu_results_dir_and_logprob(tmp_path):
    m, Y = _chain_model()
    res = m.run_gibbs(Y, nburn=3, nthin=1, nsamples=4, verbose=False, track_mu=True, results_dir=str(tmp_path))
    Mu = np.einsum('znk,zmtk->znmt', res['W'], res['V'])
    assert np.allclose(res['Mu_mean'], Mu.mean(axis=0), rtol=1e-12, atol=1e-12)
    assert os.path.exists(os.path.join(str(tmp_path), 'W.npy'))
    want = np.nansum(norm.logpdf(Y, np.einsum('nk,mtk->nmt', m.W, m.V)[..., None], np.sqrt(m.nu2)))
    assert np.isfinite(want) and np.isclose(m.logprob(Y), want, rtol=1e-13, atol=0)
    nu2 = _variances(np.random.RandomState(3))
    m.nu2, m.sample_nu2 = nu2, False
    want = GaussianLL(nu2)(Y, np.einsum('nk,mtk->nmt', m.W, m.V), m.W, m.V)
    assert np.isfinite(want) and np.isclose(m.logprob(Y), want, rtol=1e-13, atol=0)


def test_new_data_is_uploaded():
    m, Y = _chain_model()
    m.resample(Y)
    S, n_obs = m._engine.get('kappa'), m._engine.get_scalar('n_obs')
    Y2 = Y.copy()
    Y2[0, 0, 0, 0] = 5.0
    Y2[1, 1, 1] = np.nan
    m.resample(Y2)
    assert not np.array_equal(m._engine.get('kappa'), S)
    assert m._engine.get_scalar('n_obs') == np.sum(~np.isnan(Y2)) != n_obs


def test_callback_keeps_the_per_sweep_loop():
    m, Y = _chain_model()
    seen = []
    res = m.run_gibbs(Y, nburn=1, nthin=1, nsamples=2, verbose=False, callback=lambda mm, d, s, **k: seen.append(s))
    assert seen == [0, 1, 2] and res['W'].shape == (2,) + m.W.shape and res['nu2'].shape == (2, 1)


def test_held_out_scores_use_the_cell_variances():
    from functionalmf_b200.metrics import HeldOutEvaluator
    nu2 = _variances(np.random.RandomState(5), inf_frac=0.0)
    m, Y = _chain_model(R=1, nu2_true=nu2)
    target = Y[..., 0]
    train = target.copy()
    train[np.random.RandomState(6).random_sample(train.shape) < 0.15] = np.nan
    ev = HeldOutEvaluator(m, target, train=train, loglik='gaussian')
    res = m.run_gibbs(train, nburn=1, nsamples=4, verbose=False)
    Mu = np.einsum('snk,smtk->snmt', res['W'], res['V'])
    d = target[None] - Mu
    ll = -0.5 * (np.log(2 * np.pi * nu2)[None] + d * d / nu2[None])
    ps = ev.per_sample()
    for c, name in enumerate(ev.class_names):
        on = ev._classes == c
        assert on.sum() > 0
        want = ll[:, on].sum(axis=1)
        assert np.allclose(ps[:, c, 3], want, rtol=1e-10, atol=0), name


# ------------------------------------------------------------------ 4. refusals
def test_refusals():
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    from functionalmf_b200 import _lib as L
    from functionalmf_b200.engine import Engine
    m, Y = _chain_model()
    N, M, T = m.nrows, m.ncols, m.ndepth
    # invalid start: nothing changes
    W_bad = m.W.copy()
    W_bad[2] = [-1.0, 0.0, 0.0]                            # Mu decreasing in t in all of row 2
    m.W = W_bad.copy()
    V0 = m.V.copy()
    with pytest.raises(L.BTFError) as ex:
        m.resample(Y)
    assert ex.value.code == L.BTF_ESTATE and '1 row(s)' in str(ex.value)
    assert np.array_equal(m._engine.get('W'), W_bad) and np.array_equal(m._engine.get('V'), V0)
    # observed values that are not finite; nothing changes
    m2, _ = _chain_model()
    m2.resample(Y)
    S = m2._engine.get('kappa')
    Yb = Y.copy()
    Yb[0, 0, 0, 0], Yb[1, 2, 3, 1], Yb[4, 4, 4, 0] = np.inf, -np.inf, np.inf
    with pytest.raises(L.BTFError) as ex:
        m2.resample(Yb)
    assert ex.value.code == L.BTF_EINVAL and '3 observed value' in str(ex.value), str(ex.value)
    assert np.array_equal(m2._engine.get('kappa'), S)
    # per-cell variances: NaN or <= 0 at observed cells; any value at missing ones
    obs = ~np.isnan(Y).all(axis=-1)
    nu2 = np.full((N, M, T), 0.1)
    bad = nu2.copy()
    for (i, j, t), v in zip(np.argwhere(obs)[:3], (np.nan, 0.0, -1.0)):
        bad[i, j, t] = v
    m3, _ = _chain_model(nu2_true=bad)
    with pytest.raises(L.BTFError, match=r'\b3 observed cell') as ex:
        m3.resample(Y)
    assert ex.value.code == L.BTF_EINVAL
    at_missing = nu2.copy()
    at_missing[~obs] = np.nan
    m4, _ = _chain_model(nu2_true=at_missing)
    m4.resample(Y)
    # sampling nu2 while per-cell variances are set
    e = m4._engine
    e.set_nu2_cells(nu2)
    e.set_sample_mask(L.SAMPLE_ALL)
    with pytest.raises(L.BTFError) as ex:
        e.sweep(1)
    assert ex.value.code == L.BTF_ESTATE
    # the wrong upload for the engine kind
    with pytest.raises(L.BTFError) as ex:
        e.set_data_poisson(np.zeros((N, M, T)))
    assert ex.value.code == L.BTF_ESTATE
    with pytest.raises(L.BTFError) as ex:
        e.set_data_binomial(np.zeros((N, M, T)), np.ones((N, M, T)))
    assert ex.value.code == L.BTF_ESTATE
    Yc = np.ascontiguousarray(Y)
    with pytest.raises(L.BTFError) as ex:                  # (refused before the pointer is read)
        e.set_data_gaussian_rows_device(Yc.ctypes.data, 0, N, Yc.shape[3], True)
    assert ex.value.code == L.BTF_ESTATE
    for lik in (L.POISSON, L.CBINOMIAL):
        other = Engine(N, M, T, nembeds=3, tf_order=1, likelihood=lik)
        with pytest.raises(L.BTFError) as ex:
            other.set_data_gaussian(Y)
        assert ex.value.code == L.BTF_ESTATE
        other.close()
    # the other strings
    with pytest.raises(ValueError, match="'poisson', 'binomial' or 'gaussian'"):
        CM(N, M, T, 'normal', monotone(T), nembeds=3, seed=1)
    # no constraint at all (the conjugate model's job); row constraints alone are constraints
    for none in (None, np.zeros((0, 4))):
        with pytest.raises(ValueError, match='GaussianBayesianTensorFiltering'):
            CM(N, M, T, 'gaussian', np.zeros((0, T + 1)), Row_constraints=none, nembeds=3, seed=1)
    CM(N, M, T, 'gaussian', np.zeros((0, T + 1)), Row_constraints=np.array([[1.0, 0.0, 0.0, 0.0]]), nembeds=3, seed=1)
    # sharded engines
    with pytest.raises(L.BTFError) as ex:
        Engine(N, M, T, nembeds=3, tf_order=1, likelihood=L.CGAUSSIAN, world_size=2, rank=0, row_begin=0, row_end=4,
               col_begin=0, col_end=2)
    assert ex.value.code == L.BTF_EINVAL


# ------------------------------------------------------------------ 5. posterior against the host callable path
def _posterior_problem():
    rs = np.random.RandomState(8)
    N, M, T, K = 4, 3, 6, 2
    Wt = rs.uniform(0.3, 0.9, size=(N, K)); Wt[np.triu_indices(K, k=1)] = 0
    Vt = rs.uniform(0.0, 0.4, size=(M, T, K)).cumsum(axis=1)
    Y = np.einsum('nk,mtk->nmt', Wt, Vt) + 0.2 * rs.normal(size=(N, M, T))
    return N, M, T, K, Wt, Vt, Y


def _mcse_compare(summaries, names):
    (h, hs), (d, ds) = summaries
    z = (d - h) / np.sqrt(hs ** 2 + ds ** 2)
    print('posterior means of %s: max |z| %.2f' % (names, np.abs(z).max()))
    assert np.all(np.abs(z) <= 4.0), np.abs(z).max()


def _summary(m1):
    """m1 [nchains, nbatch, ...] batch means: overall mean and its MCSE (the larger of the batch and chain estimates)."""
    nchains, nbatch = m1.shape[:2]
    b = m1.reshape(nchains * nbatch, -1)
    se_b = b.std(0, ddof=1) / np.sqrt(b.shape[0])
    se_c = m1.mean(1).reshape(nchains, -1).std(0, ddof=1) / np.sqrt(nchains)
    return b.mean(0), np.maximum(se_b, se_c)


def test_posterior_matches_host_path_fixed_nu2():
    """sigma2, lam2 and Tau2 held fixed (as for the other built-in likelihoods), nu2 fixed; an EP approximation (the
    data, sd 0.3) centres the ellipses near the posterior."""
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    N, M, T, K, Wt, Vt, Y = _posterior_problem()
    nu2 = 0.04
    cons = np.concatenate([monotone(T), np.concatenate([np.eye(T), np.zeros((T, 1))], axis=1)])
    RD = CM(N, M, T, 'gaussian', cons, nembeds=K, tf_order=1, seed=1).Delta.shape[0]
    fixed = dict(sigma2_true=1.0, lam2_true=1.0, Tau2_true=np.ones((M, RD)), ep_approx=(Y, np.full(Y.shape, 0.3)))
    nburn, nsamples, nbatch, nchains = 100, 1000, 25, 4
    summaries = []
    for ll in (GaussianLL(nu2), 'gaussian'):
        m1 = np.zeros((nchains, nbatch, N, M, T))
        for c in range(nchains):
            np.random.seed(100 + c)
            m = CM(N, M, T, ll, cons, nembeds=K, tf_order=1, gass_ngrid=30, W_init=Wt, V_init=Vt * 0.8, seed=200 + c,
                   nu2_true=nu2, **fixed)
            res = m.run_gibbs(Y, nburn=nburn, nthin=1, nsamples=nsamples, verbose=False)
            Mu = np.einsum('znk,zmtk->znmt', res['W'], res['V'])
            assert np.all(np.diff(Mu, axis=-1) >= -1e-9) and np.all(Mu >= -1e-9)
            m1[c] = Mu.reshape(nbatch, -1, N, M, T).mean(axis=1)
        summaries.append(_summary(m1))
    _mcse_compare(summaries, 'Mu')


def test_posterior_matches_host_path_sampled_nu2():
    """nu2 sampled: the host loop draws nu2 from its inverse-gamma conditional given the residual of the current
    (W, V) before each host resample, which is where the engine's sweep runs its nu2 step."""
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    N, M, T, K, Wt, Vt, Y = _posterior_problem()
    cons = np.concatenate([monotone(T), np.concatenate([np.eye(T), np.zeros((T, 1))], axis=1)])
    RD = CM(N, M, T, 'gaussian', cons, nembeds=K, tf_order=1, seed=1).Delta.shape[0]
    fixed = dict(sigma2_true=1.0, lam2_true=1.0, Tau2_true=np.ones((M, RD)), ep_approx=(Y, np.full(Y.shape, 0.3)))
    a, b = 0.1, 0.1
    nburn, nsamples, nbatch, nchains = 100, 1000, 25, 4
    n_obs = np.sum(~np.isnan(Y))
    summaries = []
    for device in (False, True):
        m1 = np.zeros((nchains, nbatch, N * M * T + 1))
        for c in range(nchains):
            np.random.seed(300 + c)
            kw = dict(nembeds=K, tf_order=1, gass_ngrid=30, W_init=Wt, V_init=Vt * 0.8, seed=400 + c, **fixed)
            if device:
                m = CM(N, M, T, 'gaussian', cons, nu2_init=0.04, nu2_a=a, nu2_b=b, **kw)
                res = m.run_gibbs(Y, nburn=nburn, nthin=1, nsamples=nsamples, verbose=False)
                Mu = np.einsum('znk,zmtk->znmt', res['W'], res['V'])
                nu2s = res['nu2'][:, 0]
            else:
                ll = GaussianLL(0.04)
                m = CM(N, M, T, ll, cons, **kw)
                rs = np.random.RandomState(500 + c)
                Mu, nu2s = np.zeros((nsamples, N, M, T)), np.zeros(nsamples)
                for step in range(nburn + nsamples):
                    resid = np.nansum((Y - np.einsum('nk,mtk->nmt', m.W, m.V)) ** 2)
                    ll.nu2 = 1.0 / rs.gamma(a + n_obs / 2.0, 1.0 / (b + resid / 2.0))
                    m.resample(Y)
                    if step >= nburn:
                        Mu[step - nburn] = np.einsum('nk,mtk->nmt', m.W, m.V)
                        nu2s[step - nburn] = ll.nu2
            x = np.concatenate([Mu.reshape(nsamples, -1), nu2s[:, None]], axis=1)
            m1[c] = x.reshape(nbatch, -1, x.shape[1]).mean(axis=1)
        summaries.append(_summary(m1))
    _mcse_compare(summaries, 'Mu and nu2')
