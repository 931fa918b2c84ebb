"""Constrained model with the built-in Binomial likelihood (loglikelihood='binomial', data = (Y, Ntrials), success
probability p = W V^T): the GASS steps run inside the engine's sweep (gass_kernels.cu).  Every random choice of a
transition is a function of ngrid + 2 injected uniforms per row / column, so the device steps are compared exactly with
the host gass() driven by the same uniforms and a numpy Binomial callable."""
import os
import warnings
import numpy as np
import pytest
from scipy.stats import binom

from test_gpu_constrained_poisson import UniformRng, _device_step

pytestmark = pytest.mark.gpu


def binomial_rowcol_loglikelihood(data, WV, W, V, row=None, col=None):
    """nansum(scipy.stats.binom.logpmf(Y, Ntrials, W V^T)) over a row or a column of cells."""
    Y, Nt = data
    if row is not None:
        Y, Nt = Y[row], Nt[row]
    if col is not None:
        Y, Nt = Y[:, col], Nt[:, col]
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', category=RuntimeWarning)
        return np.nansum(binom.logpmf(Y, Nt, WV))


def box(T):
    """0 <= p <= 1 in every cell: A = [I; -I], C = [0; -1]."""
    return np.concatenate([np.concatenate([np.eye(T), -np.eye(T)]), np.concatenate([np.zeros(T), -np.ones(T)])[:, None]],
                          axis=1)


# ------------------------------------------------------------------ 1. the host gass() with the same uniforms
def _case(kind, rs):
    N, M, T, K = 8, 4, 8, 3
    W = rs.uniform(0.1, 0.6, size=(N, K))
    W[np.triu_indices(K, k=1)] = 0
    V = rs.uniform(0.05, 0.5, size=(M, T, K))
    p = np.einsum('nk,mtk->nmt', W, V)
    Nt = rs.randint(0, 21, size=p.shape).astype(float)
    Nt[rs.random_sample(p.shape) < 0.05] = 0.0            # n = 0 cells
    Y = rs.binomial(Nt.astype(int), p).astype(float)
    miss = rs.random_sample(p.shape)
    Y[miss < 0.05] = np.nan                                # NaN in Y only
    Nt[(miss >= 0.05) & (miss < 0.1)] = np.nan            # in N only
    Y[(miss >= 0.1) & (miss < 0.15)] = np.nan             # in both
    Nt[(miss >= 0.1) & (miss < 0.15)] = np.nan
    Y[3] = np.nan                                          # an all-missing row
    cons = box(T)
    kw = {}
    if kind == 'rowcons':
        kw['Row_constraints'] = np.array([[1.0, 0.0, 0.0, 0.05], [0.0, -1.0, -1.0, -1.3]])     # w_0 >= 0.05, w_1 + w_2 <= 1.3
    if kind == 'coarse':
        # no constraint at all: the coarse grid; probabilities outside [0, 1] (scipy: NaN, dropped by nansum)
        cons = np.zeros((0, T + 1))
        W = rs.normal(size=(N, K)); W[np.triu_indices(K, k=1)] = 0
        V = rs.normal(size=(M, T, K))
    if kind == 'edge':
        # p = 0 in all of row 5: y = 0 (exactly 0) except one count (-inf); p = 1 at (6, 1, 2) with y = n (exactly 0)
        # and at (4, 1, 2) with y < n (-inf)
        W[5] = 0.0
        Y[5], Nt[5] = 0.0, 10.0
        Y[5, 0, 0] = 1.0
        W[4] = W[6] = [1.0, 0.0, 0.0]
        V[1, 2] = [1.0, 0.0, 0.0]
        Nt[4, 1, 2] = Nt[6, 1, 2] = 12.0
        Y[4, 1, 2], Y[6, 1, 2] = 7.0, 12.0
    if kind == 'ep':
        p = np.einsum('nk,mtk->nmt', W, V)
        kw['ep_approx'] = (p + 0.1 * rs.normal(size=p.shape), 0.1 + 0.3 * rs.random_sample(p.shape))
    return N, M, T, K, W, V, (Y, Nt), cons, kw


CASES = [('box', 10), ('box', 40), ('box', 100), ('rowcons', 40), ('ep', 10), ('ep', 100), ('coarse', 40),
         ('edge', 40), ('edge', 11), ('slice', 40)]


@pytest.mark.parametrize('kind,ngrid', CASES)
def test_device_gass_matches_host_gass(kind, ngrid, monkeypatch):
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    from functionalmf_b200 import constrained, gass as G
    rs = np.random.RandomState(23 + ngrid + len(kind))
    N, M, T, K, W, V, data, cons, kw = _case(kind, rs)
    common = dict(nembeds=K, tf_order=1, gass_ngrid=ngrid, sigma2_init=1.0, lam2_init=0.5, W_init=W, V_init=V, seed=5,
                  **kw)
    host = CM(N, M, T, binomial_rowcol_loglikelihood, cons, **common)
    dev = CM(N, M, T, 'binomial', cons, **common)
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
        # both steps start from the initial state (a zero row of W has no active constraint, so its W step may leave
        # the constraint set, as the reference's does)
        host.W, host.V = W.copy(), V.copy()
        host._rng = UniformRng(U)
        host._sync_ep()
        if which == 'W':
            host._resample_W(data, z=zz)
        else:
            host._resample_V(data, z=zz)
        new, d = _device_step(dev, data, which, U, zz, W=W, V=V)
        ref = host.W if which == 'W' else host.V
        assert np.array_equal(d[:, 0].astype(int), np.array(log)), (d[:, 0], log)
        assert np.allclose(new, ref, rtol=1e-9, atol=1e-9), np.abs(new - ref).max()
        if kind == 'coarse':
            assert np.all(d[:, 0] == ngrid)
        if kind == 'slice':
            assert np.any(d[:, 1] == 0) or np.any(d[:, 1] < np.minimum(d[:, 0], ngrid))
        if which == 'W':
            assert np.all(new[np.triu_indices(K, k=1)] == 0)
        if kind in ('box', 'rowcons', 'ep'):
            assert not np.array_equal(new, W if which == 'W' else V)


def test_cell_log_likelihood_edges():
    """The edge cells of the 'edge' case contribute what scipy gives them, so the log-likelihood of its state is -inf
    (the device's slice test then passes every candidate) and finite once the non-matching counts are dropped."""
    rs = np.random.RandomState(1)
    N, M, T, K, W, V, (Y, Nt), cons, kw = _case('edge', rs)
    p = np.einsum('nk,mtk->nmt', W, V)
    assert binomial_rowcol_loglikelihood((Y, Nt), p, W, V) == -np.inf
    Y2 = Y.copy()
    Y2[5, 0, 0], Y2[4, 1, 2] = np.nan, np.nan
    assert np.isfinite(binomial_rowcol_loglikelihood((Y2, Nt), p, W, V))


# ------------------------------------------------------------------ 2. chains
def _chain_model(seed=11, **kw):
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    rs = np.random.RandomState(4)
    N, M, T, K = 9, 5, 12, 3
    W = rs.uniform(0.2, 0.8, size=(N, K)); W[np.triu_indices(K, k=1)] = 0
    V = rs.uniform(0.0, 0.1, size=(M, T, K)).cumsum(axis=1) / 4 + 0.02
    p = np.einsum('nk,mtk->nmt', W, V)
    Nt = np.full(p.shape, 20.0)
    Y = rs.binomial(20, p).astype(float)
    Y[rs.random_sample(Y.shape) < 0.1] = np.nan
    m = CM(N, M, T, 'binomial', box(T), nembeds=K, tf_order=1, gass_ngrid=40, W_init=W, V_init=V, seed=seed, **kw)
    return m, (Y, Nt)


def test_chain_keeps_constraints_and_is_reproducible():
    m1, data = _chain_model()
    r1 = m1.run_gibbs(data, nburn=5, nthin=2, nsamples=6, verbose=False)
    Mu = np.einsum('znk,zmtk->znmt', r1['W'], r1['V'])
    assert np.all(Mu >= 0) and np.all(Mu <= 1)
    assert not np.array_equal(r1['W'][0], r1['W'][-1])
    m2, _ = _chain_model()
    r2 = m2.run_gibbs(data, nburn=5, nthin=2, nsamples=6, verbose=False)
    for k in ('W', 'V', 'Tau2', 'sigma2', 'lam2'):
        assert np.array_equal(r1[k], r2[k]), k
    # the per-sweep loop (eager engine, one btf_sweep per resample) against run_gibbs (graph replay in segments)
    m3, _ = _chain_model(use_graph=0)
    Ws = []
    for step in range(5 + 2 * 6):
        m3.resample(data)
        if step >= 5 and (step - 5) % 2 == 0:
            Ws.append((m3.W.copy(), m3.V.copy()))
    assert np.array_equal(np.array([w for w, _ in Ws]), r1['W'])
    assert np.array_equal(np.array([v for _, v in Ws]), r1['V'])


def test_checkpoint_resumes_bit_for_bit(tmp_path):
    m, data = _chain_model()
    for _ in range(3):
        m.resample(data)
    path = str(tmp_path / 'ck.npz')
    m.save_checkpoint(path)
    ra = m.run_gibbs(data, nburn=2, nthin=1, nsamples=3, verbose=False)
    m2, _ = _chain_model()
    m2._upload(data)
    m2.load_checkpoint(path)
    rb = m2.run_gibbs(data, nburn=2, nthin=1, nsamples=3, verbose=False)
    assert np.array_equal(ra['W'], rb['W']) and np.array_equal(ra['V'], rb['V'])


def test_track_mu_results_dir_and_logprob(tmp_path):
    m, data = _chain_model()
    res = m.run_gibbs(data, nburn=3, nthin=1, nsamples=4, verbose=False, track_mu=True, results_dir=str(tmp_path))
    Mu = np.einsum('znk,zmtk->znmt', res['W'], res['V'])
    assert np.allclose(res['Mu_mean'], Mu.mean(axis=0), rtol=1e-12, atol=1e-12)
    assert os.path.exists(os.path.join(str(tmp_path), 'W.npy'))
    Y, Nt = data
    with np.errstate(all='ignore'):
        want = np.nansum(binom.logpmf(Y, Nt, np.einsum('nk,mtk->nmt', m.W, m.V)))
    assert np.isfinite(want) and m.logprob(data) == want


def test_new_data_is_uploaded():
    """Changing either array re-uploads; the chain then samples under the new data."""
    m, (Y, Nt) = _chain_model()
    m.resample((Y, Nt))
    kappa = m._engine.get('kappa')
    Y2 = Y.copy()
    Y2[0, 0, 0] = 0.0 if Y[0, 0, 0] != 0.0 else 1.0
    m.resample((Y2, Nt))
    assert not np.array_equal(m._engine.get('kappa'), kappa)
    Nt2 = Nt.copy()
    Nt2[1, 1, 1] = 25.0
    m.resample((Y2, Nt2))
    assert m._engine.get('Ntrials')[1, 1, 1] == 25.0


def test_callback_keeps_the_per_sweep_loop():
    m, data = _chain_model()
    seen = []
    res = m.run_gibbs(data, nburn=1, nthin=1, nsamples=2, verbose=False, callback=lambda mm, d, s, **k: seen.append(s))
    assert seen == [0, 1, 2] and res['W'].shape == (2,) + m.W.shape


# ------------------------------------------------------------------ 3. refusals
def test_refusals():
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    from functionalmf_b200 import NonconjugateBayesianTensorFiltering
    from functionalmf_b200 import _lib as L
    from functionalmf_b200.engine import Engine
    m, (Y, Nt) = _chain_model()
    N, M, T = m.nrows, m.ncols, m.ndepth
    # invalid start: nothing changes
    W_bad = m.W.copy()
    W_bad[2, 0] = 100.0                                    # p > 1 in all of row 2
    m.W = W_bad.copy()
    V0 = m.V.copy()
    with pytest.raises(L.BTFError) as ex:
        m.resample((Y, Nt))
    assert ex.value.code == L.BTF_ESTATE and '1 row(s)' in str(ex.value)
    assert np.array_equal(m._engine.get('W'), W_bad) and np.array_equal(m._engine.get('V'), V0)
    # counts: negative, not integers, more successes than trials; nothing changes
    m2, _ = _chain_model()
    m2.resample((Y, Nt))
    kappa = m2._engine.get('kappa')
    for edit, nbad in (({'Y': [(0, 0, 0, -1.0)]}, 1), ({'Y': [(0, 0, 1, 1.5)], 'N': [(1, 1, 1, 20.5)]}, 2),
                       ({'Y': [(2, 0, 0, 21.0), (2, 0, 1, 30.0), (2, 0, 2, 20.0)]}, 2), ({'N': [(3, 1, 0, -1.0)]}, 1)):
        Yb, Nb = np.where(np.isnan(Y), 0.0, Y), Nt.copy()
        for name, arr in (('Y', Yb), ('N', Nb)):
            for i, j, t, v in edit.get(name, []):
                arr[i, j, t] = v
        with pytest.raises(L.BTFError) as ex:
            m2.resample((Yb, Nb))
        assert ex.value.code == L.BTF_EINVAL and '%d observed cell' % nbad in str(ex.value), str(ex.value)
        assert np.array_equal(m2._engine.get('kappa'), kappa)
    # a bad count in a missing cell is not a count
    Yb, Nb = Y.copy(), Nt.copy()
    Yb[0, 0, 0], Nb[0, 0, 0] = -3.0, np.nan
    m2.resample((Yb, Nb))
    # data that are not two [N, M, T] arrays
    for bad in (Y, (Y,), (Y, Nt, Nt), (Y[:-1], Nt[:-1]), (Y, Nt[..., None])):
        with pytest.raises(ValueError):
            m2.resample(bad)
    # the wrong upload for the engine kind
    with pytest.raises(L.BTFError) as ex:
        m2._engine.set_data_poisson(np.zeros((N, M, T)))
    assert ex.value.code == L.BTF_ESTATE
    with pytest.raises(L.BTFError) as ex:
        m2._engine.set('Ntrials', Nt)
    assert ex.value.code == L.BTF_ESTATE
    ep = Engine(N, M, T, nembeds=3, tf_order=1, likelihood=L.POISSON)
    with pytest.raises(L.BTFError) as ex:
        ep.set_data_binomial(Y, Nt)
    assert ex.value.code == L.BTF_ESTATE
    # the other strings
    with pytest.raises(ValueError):
        CM(N, M, T, 'binom', box(T), nembeds=3, seed=1)
    with pytest.raises(ValueError):
        NonconjugateBayesianTensorFiltering(N, M, T, 'binomial', nembeds=3, seed=1)
    # sharded engines
    with pytest.raises(L.BTFError) as ex:
        Engine(N, M, T, nembeds=3, tf_order=1, likelihood=L.CBINOMIAL, world_size=2, rank=0, row_begin=0, row_end=4,
               col_begin=0, col_end=2)
    assert ex.value.code == L.BTF_EINVAL


# ------------------------------------------------------------------ 4. posterior against the host callable path
def test_posterior_matches_host_path():
    """sigma2, lam2 and Tau2 are held fixed: with them sampled, this tiny problem's hyper-parameters drift (the scale of
    W V^T is shared between W and V), so two chains agree only while they are equally long.  Fixed, both paths sample
    one stationary posterior of W and V, and equally long chains of the host and device GASS steps must agree.  An EP
    approximation (the observed fractions, sd 0.15) centres the ellipses near that posterior, so that 1000 samples
    per chain measure its mean to within a few MCSE; centred on the prior, some entries mix too slowly for that."""
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    rs = np.random.RandomState(8)
    N, M, T, K = 4, 3, 6, 2
    Wt = rs.uniform(0.3, 0.9, size=(N, K)); Wt[np.triu_indices(K, k=1)] = 0
    Vt = rs.uniform(0.05, 0.5, size=(M, T, K))
    Nt = np.full((N, M, T), 15.0)
    Y = rs.binomial(15, np.einsum('nk,mtk->nmt', Wt, Vt)).astype(float)
    data = (Y, Nt)
    RD = CM(N, M, T, 'binomial', box(T), nembeds=K, tf_order=1, seed=1).Delta.shape[0]
    fixed = dict(sigma2_true=1.0, lam2_true=1.0, Tau2_true=np.ones((M, RD)), ep_approx=(Y / Nt, np.full(Y.shape, 0.15)))
    nburn, nsamples, nbatch, nchains = 100, 1000, 25, 4
    summaries = []
    for ll in (binomial_rowcol_loglikelihood, 'binomial'):
        m1 = np.zeros((nchains, nbatch, N, M, T))
        for c in range(nchains):
            np.random.seed(100 + c)
            m = CM(N, M, T, ll, box(T), nembeds=K, tf_order=1, gass_ngrid=30, W_init=Wt, V_init=Vt * 0.8, seed=200 + c,
                   **fixed)
            res = m.run_gibbs(data, nburn=nburn, nthin=1, nsamples=nsamples, verbose=False)
            Mu = np.einsum('znk,zmtk->znmt', res['W'], res['V'])
            assert np.all(Mu >= 0) and np.all(Mu <= 1)
            m1[c] = Mu.reshape(nbatch, -1, N, M, T).mean(axis=1)
        b = m1.reshape(nchains * nbatch, -1)
        se_b = b.std(0, ddof=1) / np.sqrt(b.shape[0])
        se_c = m1.mean(1).reshape(nchains, -1).std(0, ddof=1) / np.sqrt(nchains)
        summaries.append((b.mean(0), np.maximum(se_b, se_c)))
    (h, hs), (d, ds) = summaries
    z = (d - h) / np.sqrt(hs ** 2 + ds ** 2)
    frac = float(np.mean(np.abs(z) <= 4.0))
    print('posterior mean of Mu: %.4f of entries within 4 MCSE (max |z| %.2f)' % (frac, np.abs(z).max()))
    assert frac >= 0.99, frac
