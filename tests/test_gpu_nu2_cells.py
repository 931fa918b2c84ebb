"""Gaussian model with known per-cell noise variances (nu2 an [N, M, T] array, the reference's heteroskedastic
branch): one sweep against the CPU oracle, +inf as missing, the scalar special case, the reference's semantics
of a sampled nu2, rejections, run_gibbs / checkpoint / graph behaviour, the integer statistics path and the
held-out scores.  Run on the B200 box: pytest -m gpu."""
import numpy as np
import pytest

from golden_util import relerr, normerr
from gpu_util import band_rows_from_lower, load_state, inject_all
from test_gpu_parity import SHAPES, _random_problem, _random_state, _random_noise

pytestmark = pytest.mark.gpu

TOL = 1e-10
EPS = np.finfo(float).eps
NO_NU2 = 127 & ~1          # every step but the nu2 step


def _variances(rs, Y, n_inf=0.05):
    """nu2 = gamma + 0.1, with +inf at a share of the observed cells (missing cells keep finite values)."""
    obs = ~np.isnan(Y).all(axis=-1) if Y.ndim == 4 else ~np.isnan(Y)
    nu2 = rs.gamma(2.0, size=obs.shape) + 0.1
    nu2[obs & (rs.random_sample(obs.shape) < n_inf)] = np.inf
    return nu2


def _check_v(eng, O, W, st, noise, cw, sw, Delta, lam2, Tau2, order):
    Vn, dV = O.step_V(W, st['V'], cw, sw, Delta, lam2, Tau2, noise['z_V'], order, want_diag=True)
    band, mean, Vg = eng.diag('V_band'), eng.diag('V_mean'), eng.get('V')
    for j in range(Vg.shape[0]):
        assert normerr(band[j], band_rows_from_lower(dV['band'][j])) < TOL, j
        Qd = O.band_to_dense_lower(dV['band'][j])
        Qd = Qd + np.tril(Qd, -1).T
        tol = max(TOL, 50 * np.linalg.cond(Qd) * EPS)
        assert normerr(mean[j], dV['mean'][j]) < tol, j
        assert normerr(Vg[j], Vn[j]) < tol, j


# 3-D (R = 1) and 4-D data, K = 1, 5, 8, 16, 17, 32, orders 0-3, forced statistics splits
SUBSET = [SHAPES[i] for i in (1, 3, 5, 6, 7, 8)]


@pytest.mark.parametrize('shape', SUBSET)
def test_sweep_with_cell_variances_vs_oracle(shape):
    from oracle import btf_oracle as O
    from functionalmf_b200.engine import Engine
    N, M, T, R, K, order, opts = shape
    rs = np.random.RandomState(2000 + N + K)
    W, V, Y = _random_problem(rs, N, M, T, R, K)
    if R == 1:
        Y = Y[..., 0]
    nu2 = _variances(rs, Y)
    eng = Engine(N, M, T, nembeds=K, tf_order=order, seed=5, **opts)
    Delta = eng.get('Delta')
    st = _random_state(rs, N, M, T, K, Delta.shape[0], W, V)
    noise = _random_noise(rs, N, M, T, K, Delta.shape[0])
    noise.pop('g_nu2')
    eng.set_data_gaussian(Y)
    eng.set_nu2_cells(nu2)
    eng.set_sample_mask(NO_NU2)
    eng.enable_diag(True)
    load_state(eng, st)
    inject_all(eng, noise)
    eng.sweep(1)
    cnt, S, _ = O.prereduce(Y)
    cw, sw = O.gaussian_weights(cnt, S, nu2)
    Lp = K * (K + 1) // 2
    il = np.tril_indices(K)
    A, b = O.row_stats(st['V'], cw, sw)
    rstat = eng.diag('row_stats')
    assert normerr(rstat[:, :Lp], A[:, il[0], il[1]]) < TOL
    assert normerr(rstat[:, Lp:], b) < TOL
    cfg = dict(K=K, order=order, Delta=Delta, nu2_a=0.1, nu2_b=0.1, sigma2_a=0.1, sigma2_b=0.1, stability=1e-6,
               force_psd=True, force_psd_eps=1e-6, force_psd_attempts=4, ref_compat=True, sample_nu2=False)
    want = O.gaussian_sweep(dict(st, nu2=nu2), Y, noise, cfg)
    Ac, bc = O.col_stats(want['W'], cw, sw)
    cstat = eng.diag('col_stats')
    assert normerr(cstat[:, :Lp], Ac.reshape(M * T, K, K)[:, il[0], il[1]]) < TOL
    assert normerr(cstat[:, Lp:], bc.reshape(M * T, K)) < TOL
    for k in ('sigma2', 'lam2', 'lam2_a'):
        assert relerr(eng.get_scalar(k), want[k]) < TOL, k
    for k in ('Tau2', 'Tau2_a', 'Tau2_b', 'Tau2_c'):
        assert relerr(eng.get(k), want[k]) < TOL, k
    assert normerr(eng.get('W'), want['W']) < 1e-9
    _check_v(eng, O, want['W'], st, noise, cw, sw, Delta, want['lam2'], want['Tau2'], order)
    eng.close()


def _problem(seed=3, N=90, M=7, T=12, R=2, K=5, nan_frac=0.2):
    rs = np.random.RandomState(seed)
    W, V, Y = _random_problem(rs, N, M, T, R, K, nan_frac)
    return rs, Y, _variances(rs, Y, n_inf=0.0)


def _model(Y, K=5, seed=7, **kw):
    from functionalmf_b200.factor import GaussianBayesianTensorFiltering as G
    N, M, T = Y.shape[:3]
    return G(N, M, T, nembeds=K, tf_order=2, seed=seed, **kw)


def _chain(m, Y, n):
    out = []
    for _ in range(n):
        m.resample(Y)
        out.append((m.W.copy(), m.V.copy(), m.Tau2.copy()))
    return out


def _same_chains(a, b):
    for x, y in zip(a, b):
        for u, v in zip(x, y):
            assert np.array_equal(u, v)


def test_infinite_variance_is_exactly_missing():
    rs, Y, nu2 = _problem()
    obs = ~np.isnan(Y).all(axis=-1)
    hole = obs & (rs.random_sample(obs.shape) < 0.1)
    nu2_inf = nu2.copy()
    nu2_inf[hole] = np.inf
    Y_nan = Y.copy()
    Y_nan[hole] = np.nan
    a = _model(Y, nu2_true=nu2_inf).run_gibbs(Y, nburn=0, nsamples=5, verbose=False)
    b = _model(Y_nan, nu2_true=nu2_inf).run_gibbs(Y_nan, nburn=0, nsamples=5, verbose=False)
    for k in ('W', 'V', 'Tau2'):
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize('c, v_tol', [(0.5, TOL), (0.7, 1e-9)])
def test_constant_variances_equal_the_scalar(monkeypatch, c, v_tol):
    # per-cell weights cnt / c against statistics scaled by 1 / c afterwards: exact for a power of two; otherwise the
    # rounding differs and the band solve's conditioning carries it through the chain (1.7e-10 in V after 3 sweeps
    # at c = 0.7 on a B200, with W within 1e-10)
    monkeypatch.setenv('BTF_STATS_NO_I8', '1')
    _, Y, _ = _problem()
    a = _model(Y, nu2_true=np.full(Y.shape[:3], c))
    b = _model(Y, nu2_true=c)
    for (wa, va, _), (wb, vb, _) in zip(_chain(a, Y, 3), _chain(b, Y, 3)):
        assert normerr(wa, wb) < TOL
        assert normerr(va, vb) < v_tol


def test_sampled_nu2_follows_the_reference():
    from oracle import btf_oracle as O
    rs, Y, nu2 = _problem()
    # nu2_init = array with sample_nu2 True: the nu2 step draws a scalar from the residual; the array is never used
    m = _model(Y, nu2_init=nu2)
    assert m.sample_nu2 and m.nu2.shape == nu2.shape
    g = 37.5
    want = O.step_nu2(m.W, m.V, Y, 0.1, 0.1, g)[0]
    m._engine.inject('g_nu2', [g])
    m.resample(Y)
    assert np.ndim(m.nu2) == 0 and relerr(m.nu2, want) < TOL
    # two per-cell sweeps, then sample_nu2 = True: the next sweep recomputes the residual (no weighted by-product)
    m = _model(Y, nu2_true=nu2)
    _chain(m, Y, 2)
    assert m.nu2 is not None and np.shape(m.nu2) == nu2.shape
    m.sample_nu2 = True
    Delta = m._engine.get('Delta')
    noise = _random_noise(rs, *Y.shape[:3], 5, Delta.shape[0])
    st = dict(W=m.W.copy(), V=m.V.copy(), Tau2=m.Tau2.copy(), Tau2_a=m.Tau2_a.copy(), Tau2_b=m.Tau2_b.copy(),
              Tau2_c=m.Tau2_c.copy(), lam2=m.lam2, lam2_a=m.lam2_a, sigma2=m.sigma2, nu2=1.0)
    cfg = dict(K=5, order=2, Delta=Delta, nu2_a=0.1, nu2_b=0.1, sigma2_a=0.1, sigma2_b=0.1, stability=1e-6,
               force_psd=True, force_psd_eps=1e-6, force_psd_attempts=4, ref_compat=True)
    want = O.gaussian_sweep(st, Y, noise, cfg)
    inject_all(m._engine, noise)
    m.resample(Y)
    assert np.ndim(m.nu2) == 0
    for k in ('nu2', 'sigma2', 'lam2', 'lam2_a'):
        assert relerr(getattr(m, k), want[k]) < TOL, k
    assert relerr(m.Tau2, want['Tau2']) < TOL
    assert normerr(m.W, want['W']) < 1e-9
    assert normerr(m.V, want['V']) < 1e-6


def test_bad_variances_are_refused():
    from functionalmf_b200.engine import Engine
    from functionalmf_b200 import _lib as L
    _, Y, nu2 = _problem()
    N, M, T = Y.shape[:3]
    obs = ~np.isnan(Y).all(axis=-1)
    oi, mi = np.argwhere(obs), np.argwhere(~obs)
    bad_vals = [np.nan, np.nan, -1.0, 0.0, -np.inf]
    eng = Engine(N, M, T, nembeds=5, tf_order=2, seed=1)
    eng.set_data_gaussian(Y)
    eng.init_state(127)
    eng.set_sample_mask(NO_NU2)
    at_missing = nu2.copy()
    for (i, j, t), v in zip(mi, bad_vals):
        at_missing[i, j, t] = v
    eng.set_nu2_cells(at_missing)             # any value at a missing cell is accepted
    eng.sweep(1)
    at_obs = nu2.copy()
    for (i, j, t), v in zip(oi, bad_vals):
        at_obs[i, j, t] = v
    with pytest.raises(L.BTFError, match=r'\b5 observed cell') as ei:
        eng.set_nu2_cells(at_obs)
    assert ei.value.code == L.BTF_EINVAL
    # the engine fell back to the scalar nu2, and a sweep with the nu2 step runs
    eng.set_sample_mask(127)
    eng.sweep(1)
    # new data that observes the bad cells of accepted variances: refused at the next sweep
    eng.set_nu2_cells(at_missing)
    eng.set_sample_mask(NO_NU2)
    Y2 = np.where(np.isnan(Y), 0.5, Y)
    eng.set_data_gaussian(Y2)
    with pytest.raises(L.BTFError, match=r'\b5 observed cell') as ei:
        eng.sweep(1)
    assert ei.value.code == L.BTF_EINVAL
    # the nu2 step cannot run with per-cell variances
    eng.set_data_gaussian(Y)
    eng.sweep(1)
    eng.set_sample_mask(127)
    with pytest.raises(L.BTFError) as ei:
        eng.sweep(1)
    assert ei.value.code == L.BTF_ESTATE
    eng.close()
    # the model classes: the same count, and ValueError for a wrong shape
    m = _model(Y, nu2_true=at_obs)
    with pytest.raises(L.BTFError, match=r'\b5 observed cell'):
        m.resample(Y)
    m = _model(Y, nu2_true=nu2)
    m.nu2 = np.ones((N, M))
    with pytest.raises(ValueError):
        m.resample(Y)
    m.sample_nu2 = True
    with pytest.raises(ValueError):
        m.resample(Y)
    # non-Gaussian engines and sharded engines
    for lik in (L.BINOMIAL, L.NEGBINOMIAL):
        e = Engine(N, M, T, nembeds=5, tf_order=2, likelihood=lik)
        with pytest.raises(L.BTFError) as ei:
            e.set_nu2_cells(nu2)
        assert ei.value.code == L.BTF_ESTATE
        e.close()
    e = Engine(N, M, T, nembeds=5, tf_order=2, world_size=2, rank=0, row_begin=0, row_end=N // 2, col_begin=0,
               col_end=M // 2)
    with pytest.raises(L.BTFError) as ei:
        e.set_nu2_cells(nu2[:N // 2])
    assert ei.value.code == L.BTF_EINVAL
    e.close()


def test_run_gibbs_and_mode_switches(tmp_path):
    _, Y, nu2 = _problem()
    nburn, nthin, nsamples = 2, 2, 3
    a = _model(Y, nu2_true=nu2)
    res = a.run_gibbs(Y, nburn=nburn, nthin=nthin, nsamples=nsamples, verbose=True, print_freq=3)
    b = _model(Y, nu2_true=nu2)
    loop = _chain(b, Y, nburn + nthin * nsamples)[nburn::nthin]
    for s, (w, v, t) in enumerate(loop):
        assert np.array_equal(res['W'][s], w) and np.array_equal(res['V'][s], v) and np.array_equal(res['Tau2'][s], t)
    assert res['nu2'].shape == (nsamples,) + nu2.shape and not res['nu2'].flags.writeable
    assert np.array_equal(res['nu2'], np.broadcast_to(nu2, res['nu2'].shape))
    # per-cell -> scalar -> per-cell on one model == fresh models from the same state
    for k, fixed in enumerate((1.3, nu2)):
        a.nu2 = fixed
        path = str(tmp_path / ('s%d.npz' % k))
        a.save_checkpoint(path)
        f = _model(Y, nu2_true=fixed)
        f.load_checkpoint(path)
        f.nu2 = fixed
        ra = a.run_gibbs(Y, nburn=1, nsamples=3, verbose=False)
        rf = f.run_gibbs(Y, nburn=1, nsamples=3, verbose=False)
        for key in ('W', 'V', 'Tau2'):
            assert np.array_equal(ra[key], rf[key]), (k, key)
        assert ra['nu2'].shape == ((3, 1) if k == 0 else (3,) + nu2.shape)


def test_integer_statistics_path_is_not_taken(monkeypatch, tmp_path):
    from functionalmf_b200 import _lib as L
    rs = np.random.RandomState(8)
    W, V, Y = _random_problem(rs, 300, 20, 16, 3, 16)
    nu2 = _variances(rs, Y)
    monkeypatch.setenv('BTF_STATS_FORCE_I8', '1')
    a = _model(Y, K=16, nu2_true=nu2)
    ca = _chain(a, Y, 2)
    assert list(a._engine.diag('i8_route')) == [0, 0]          # per-cell sweeps ran the FP64 statistics
    monkeypatch.delenv('BTF_STATS_FORCE_I8')
    _same_chains(ca, _chain(_model(Y, K=16, nu2_true=nu2), Y, 2))
    monkeypatch.setenv('BTF_STATS_FORCE_I8', '1')
    a.nu2 = 0.9
    path = str(tmp_path / 'i8.npz')
    a.save_checkpoint(path)
    b = _model(Y, K=16, nu2_true=0.9)
    b.load_checkpoint(path)
    b.nu2 = 0.9
    _same_chains(_chain(a, Y, 3), _chain(b, Y, 3))
    for m in (a, b):
        assert set(m._engine.diag('i8_route')) <= {L.I8_ROUTE_FUSED, L.I8_ROUTE_SPLITK}
        assert min(m._engine.diag('i8_route')) > 0


def test_checkpoint_resumes_bit_for_bit(tmp_path):
    _, Y, nu2 = _problem()
    a = _model(Y, nu2_true=nu2)
    _chain(a, Y, 2)
    path = str(tmp_path / 'ck.npz')
    a.save_checkpoint(path)
    b = _model(Y, nu2_true=nu2)
    b.load_checkpoint(path)
    _same_chains(_chain(a, Y, 3), _chain(b, Y, 3))


def test_held_out_scores_use_the_cell_variances():
    from scipy.special import erfc
    from functionalmf_b200.metrics import HeldOutEvaluator
    rs, Y, nu2 = _problem(R=1, nan_frac=0.1)
    target = Y[..., 0]
    train = target.copy()
    train[rs.random_sample(train.shape) < 0.15] = np.nan
    m = _model(train, nu2_true=nu2)
    ev = HeldOutEvaluator(m, target, train=train, loglik='gaussian', predictive=True)
    res = m.run_gibbs(train, nburn=1, nsamples=4, verbose=False)
    cls = ev._classes
    Mu = np.einsum('snk,smtk->snmt', res['W'], res['V'])
    d = target[None] - Mu
    ll = -0.5 * (np.log(2 * np.pi * nu2)[None] + d * d / nu2[None])
    ps = ev.per_sample()
    mean = Mu.mean(axis=0)
    dm = target - mean
    llm = -0.5 * (np.log(2 * np.pi * nu2) + dm * dm / nu2)
    F = (0.5 * erfc(-(d / np.sqrt(nu2)[None]) / np.sqrt(2))).mean(axis=0)
    nll = ev.nll_of_mean()
    summ = ev._summary(pred_lo=0.025, pred_hi=0.975)
    for c, name in enumerate(ev.class_names):
        on = cls == c
        assert on.sum() > 0
        assert relerr(ps[:, c, 3], ll[:, on].sum(axis=1)) < TOL, name
        assert relerr(-nll[name], llm[on].sum()) < TOL, name
        assert summ[c, 5] == np.sum((F[on] >= 0.025) & (F[on] <= 0.975)), name
