"""Constrained model with the built-in Poisson likelihood (loglikelihood='poisson'): the GASS steps run inside the
engine's sweep (gass_kernels.cu).  Every random choice of a transition is a function of ngrid + 2 injected uniforms
per row / column, so the device steps are compared exactly with the reference's recorded workers
(oracle/make_golden_constrained.py) and with the host gass() driven by the same uniforms."""
import os
import numpy as np
import pytest
from scipy.stats import poisson

from golden_util import GOLDEN
from constrained_ll import rowcol_loglikelihood, ReplayRng
from test_gass_host import unpack_choices

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------ helpers
class UniformRng(object):
    """np.random stand-in that turns one row of uniforms [slice, ngrid thinning, pick] per gass() call into the host
    transition the device takes: the thinning is the partial Fisher-Yates over the ascending feasible grid."""

    def __init__(self, U):
        self.U, self.row, self.G = np.asarray(U), -1, {}

    def random(self, size=None):
        self.row += 1
        return self.U[self.row, 0]

    def choice(self, a, size=None, replace=True):
        u = self.U[self.row]
        if size is None:
            self.G[self.row] = a
            return min(int(np.floor(u[-1] * a)), a - 1)
        lst = list(np.asarray(a))
        F = len(lst)
        for k in range(size):
            r = min(k + int(np.floor(u[1 + k] * (F - k))), F - 1)
            lst[k], lst[r] = lst[r], lst[k]
        return np.array(lst[:size])


class TapeToUniforms(object):
    """Replays a recorded reference tape and writes down the uniforms that make the device take the same choices."""

    def __init__(self, uniforms, choices, ngrid):
        self.tape = ReplayRng(uniforms, choices)
        self.ngrid, self.rows = ngrid, []

    def random(self, size=None):
        u = self.tape.random()
        self.rows.append(np.full(self.ngrid + 2, 0.5))
        self.rows[-1][0] = u
        return u

    def choice(self, a, size=None, replace=True):
        c = self.tape.choice(a, size, replace)
        row = self.rows[-1]
        if size is None:
            row[-1] = (int(c) + 0.5) / a
            return c
        lst = list(np.asarray(a))
        F = len(lst)
        for k, ang in enumerate(np.asarray(c)):
            r = k + lst[k:].index(ang)
            row[1 + k] = (r - k + 0.5) / (F - k)
            lst[k], lst[r] = lst[r], lst[k]
        return c


def _models(z, with_ep, **kw):
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    N, M, T, K, order, ngrid = [int(x) for x in z['dims']]
    sigma2, lam2, stab = [float(x) for x in z['scal']]
    args = dict(ep_approx=(z['Mu_ep'], z['Sigma_ep']) if with_ep else None, nembeds=K, tf_order=order, gass_ngrid=ngrid,
                sigma2_init=sigma2, lam2_init=lam2, Tau2_init=z['Tau2'], W_init=z['W0'], V_init=z['V0'], stability=stab,
                seed=3)
    args.update(kw)
    host = CM(N, M, T, rowcol_loglikelihood, z['Constraints'], **args)
    dev = CM(N, M, T, 'poisson', z['Constraints'], **args)
    return host, dev


def _device_step(m, Y, which, U, zz, W=None, V=None):
    """One W-only or V-only device sweep with injected uniforms and normals; returns (state, diag)."""
    from functionalmf_b200 import _lib as L
    if W is not None:
        m.W = np.array(W, dtype=float)
    if V is not None:
        m.V = np.array(V, dtype=float)
    m._begin(Y)
    eng = m._engine
    eng.set_sample_mask(L.SAMPLE_W if which == 'W' else L.SAMPLE_V)
    eng.inject('gass_u_' + which, U)
    eng.inject('z_' + which, zz)
    eng.enable_diag(True)
    eng.sweep(1)
    d = eng.diag('gass_' + which)
    eng.enable_diag(False)
    return eng.get(which), d


# ------------------------------------------------------------------ 1. the reference's recorded workers
@pytest.mark.parametrize('name,with_ep', [('constrained_plain', False), ('constrained_ep', True)])
def test_device_gass_matches_reference_workers(name, with_ep):
    z = np.load(os.path.join(GOLDEN, name + '.npz'))
    ngrid = int(z['dims'][5])
    host, dev = _models(z, with_ep)
    Y = z['Y']
    host._sync_ep()
    host._rng = TapeToUniforms(z['W_u'], unpack_choices(z['W_c'], z['W_clen']), ngrid)
    host._resample_W(Y, z=z['W_z'])
    UW = np.array(host._rng.rows)
    host.W[:] = z['W1']
    host._rng = TapeToUniforms(z['V_u'], unpack_choices(z['V_c'], z['V_clen']), ngrid)
    host._resample_V(Y, z=z['V_z'])
    UV = np.array(host._rng.rows)
    W1, _ = _device_step(dev, Y, 'W', UW, z['W_z'], W=z['W0'], V=z['V0'])
    assert np.allclose(W1, z['W1'], rtol=1e-9, atol=1e-11), np.abs(W1 - z['W1']).max()
    V1, _ = _device_step(dev, Y, 'V', UV, z['V_z'], W=z['W1'], V=z['V0'])
    assert np.allclose(V1, z['V1'], rtol=1e-7, atol=1e-9), np.abs(V1 - z['V1']).max()


# ------------------------------------------------------------------ 2. the host gass() with the same uniforms
def _case(kind, ngrid, rs):
    N, M, T, K, R = 7, 4, 8, 3, 2
    W = np.abs(rs.normal(size=(N, K))) + 0.1
    W[np.triu_indices(K, k=1)] = 0
    V = np.abs(rs.normal(size=(M, T, K))) + 0.1
    lam = np.einsum('nk,mtk->nmt', W, V)
    Y = rs.poisson(lam[..., None] * np.ones(R)).astype(float)
    Y[rs.random_sample(Y.shape) < 0.2] = np.nan
    Y[3] = np.nan                                  # an all-missing row
    cons = np.concatenate([np.eye(T), np.zeros((T, 1))], axis=1)     # Mu >= 0
    kw = {}
    if kind == 'rowcons':
        kw['Row_constraints'] = np.array([[1.0, 0.0, 0.0, 0.05], [0.0, 1.0, 1.0, -5.0]])
    if kind == 'empty':
        # w_0 >= 0.5 and w_1 >= -0.3 met with equality: with a proposal v_0, v_1 > 0 (z_W > 0, no EP) the feasible arcs
        # are [0, 2 atan(v_0 / 0.5)] and [-2 atan(v_1 / 0.3), 0], so after the EDGE_EPS shrink the grid of rows i >= 1
        # is empty; no tensor constraints (the rates may go negative)
        W[:, 0] = 0.5
        W[1:, 1] = -0.3
        cons = np.zeros((0, T + 1))
        kw['Row_constraints'] = np.array([[1.0, 0.0, 0.0, 0.5], [0.0, 1.0, 0.0, -0.3]])
    if kind == 'coarse':
        # no constraint at all: the coarse grid; negative rates (scipy: NaN, dropped by nansum)
        cons = np.zeros((0, T + 1))
        W = rs.normal(size=(N, K)); W[np.triu_indices(K, k=1)] = 0
        V = rs.normal(size=(M, T, K))
    if kind == 'zero_rate':
        W[5] = 0.0                                 # lambda = 0 with y > 0 in row 5: ll = -inf
        Y[5] = 2.0
    if kind == 'ep':
        kw['ep_approx'] = (lam + 0.3 * rs.normal(size=lam.shape), 0.5 + rs.random_sample(lam.shape))
    return N, M, T, K, W, V, Y, cons, kw


CASES = [('plain', 10), ('plain', 40), ('plain', 100), ('rowcons', 40), ('ep', 10), ('ep', 100), ('empty', 40),
         ('coarse', 40), ('zero_rate', 40), ('slice', 40)]


@pytest.mark.parametrize('kind,ngrid', CASES)
def test_device_gass_matches_host_gass(kind, ngrid, monkeypatch):
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    from functionalmf_b200 import constrained, gass as G
    rs = np.random.RandomState(17 + ngrid + len(kind))
    N, M, T, K, W, V, Y, cons, kw = _case(kind, ngrid, rs)
    common = dict(nembeds=K, tf_order=1, gass_ngrid=ngrid, sigma2_init=1.0, lam2_init=0.5, W_init=W, V_init=V, seed=5,
                  **kw)
    host = CM(N, M, T, rowcol_loglikelihood, cons, **common)
    dev = CM(N, M, T, 'poisson', cons, **common)
    log = []

    def recording_gass(x, v, ll, Cons, mu=None, ll_args=None, ngrid=100, rng=None):
        mu_ = np.zeros_like(x) if mu is None else mu
        A, c = Cons[:, :-1], Cons[:, -1]
        a, b, cc = A.dot(x - mu_), A.dot(v), c - A.dot(mu_)
        F = len(G.feasible_angles(a, b, cc, ngrid))
        disc = a ** 2 + b ** 2 - cc ** 2
        act = (disc >= 0) & (a != -cc)
        roots = np.concatenate([2 * np.arctan((b[act] + np.sqrt(disc[act])) / (a + cc)[act]),
                                2 * np.arctan((b[act] - np.sqrt(disc[act])) / (a + cc)[act])])
        cur = ll(x, ll_args)
        height = cur + np.log(rng.U[rng.row + 1, 0])
        out = G.gass(x, v, ll, Cons, mu=mu, cur_ll=cur, ll_args=ll_args, ngrid=ngrid, rng=rng)
        log.append(dict(F=F, height=height, roots=roots, new_ll=out[1]))
        return out
    monkeypatch.setattr(constrained, 'gass', recording_gass)

    # (zero_rate: a zero row of W has no active constraint, so its W step may leave the constraint set, as the
    #  reference's does; only the V step is compared)
    for which in (('V',) if kind == 'zero_rate' else ('W', 'V')):
        n = N if which == 'W' else M
        U = rs.random_sample((n, ngrid + 2))
        if kind == 'slice':
            U[:, 0] = 1.0 - 1e-16          # height = current ll: often no candidate clears it
        zz = rs.normal(size=(N, K) if which == 'W' else (M, T, K))
        if kind == 'empty' and which == 'W':
            zz = np.abs(zz) + 0.1
        del log[:]
        host.W, host.V = dev.W.copy(), dev.V.copy()
        host._rng = UniformRng(U)
        host._sync_ep()
        if which == 'W':
            host._resample_W(Y, z=zz)
        else:
            host._resample_V(Y, z=zz)
        new, d = _device_step(dev, Y, which, U, zz)
        ref = host.W if which == 'W' else host.V
        F = np.array([r['F'] for r in log])
        ok_F = np.array_equal(d[:, 0].astype(int), F)
        ok_x = np.allclose(new, ref, rtol=1e-9, atol=1e-9)
        if not (ok_F and ok_x):
            for i, r in enumerate(log):
                grid = np.linspace(-np.pi, np.pi, G.FINE_GRID)
                dist = np.min(np.abs(grid[:, None] - r['roots'][None])) if r['roots'].size else np.inf
                print('%s %d: F host %d device %d, G host %d device %d, theta %.6f, host |ll - height| %.3e, '
                      'closest root to a grid point %.3e, max |x_host - x_device| %.3e'
                      % (which, i, r['F'], d[i, 0], host._rng.G.get(i, 0), d[i, 1], d[i, 2],
                         abs(r['new_ll'] - r['height']), dist, np.abs(new[i] - ref[i]).max()))
        assert ok_F, (d[:, 0], F)
        assert ok_x, np.abs(new - ref).max()
        if kind == 'empty' and which == 'W':
            assert np.all(d[1:, 0] == 0) and np.array_equal(new[1:], W[1:]) and d[0, 0] > 0
        if kind == 'coarse':
            assert np.all(d[:, 0] == ngrid)
        if which == 'W':
            assert np.all(new[np.triu_indices(K, k=1)] == 0)
        dev.W, dev.V = new if which == 'W' else dev.W, new if which == 'V' else dev.V


# ------------------------------------------------------------------ 3. chains
def _chain_model(seed=11, **kw):
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    rs = np.random.RandomState(4)
    N, M, T, K = 9, 5, 12, 3
    W = np.abs(rs.normal(size=(N, K))) + 0.1; W[np.triu_indices(K, k=1)] = 0
    V = np.abs(rs.normal(size=(M, T, K))).cumsum(axis=1) * 0.3 + 0.1
    Y = rs.poisson(np.einsum('nk,mtk->nmt', W, V)).astype(float)
    Y[rs.random_sample(Y.shape) < 0.1] = np.nan
    cons = np.concatenate([np.eye(T), np.zeros((T, 1))], axis=1)
    m = CM(N, M, T, 'poisson', cons, nembeds=K, tf_order=1, gass_ngrid=40, W_init=W, V_init=V, seed=seed,
           **kw)
    return m, Y


def test_chain_keeps_constraints_and_is_reproducible():
    m1, Y = _chain_model()
    r1 = m1.run_gibbs(Y, nburn=5, nthin=2, nsamples=6, verbose=False)
    Mu = np.einsum('znk,zmtk->znmt', r1['W'], r1['V'])
    assert np.all(Mu >= 0)
    assert not np.array_equal(r1['W'][0], r1['W'][-1])
    m2, _ = _chain_model()
    r2 = m2.run_gibbs(Y, nburn=5, nthin=2, nsamples=6, verbose=False)
    for k in ('W', 'V', 'Tau2', 'sigma2', 'lam2'):
        assert np.array_equal(r1[k], r2[k]), k
    # the per-sweep loop (eager engine, one btf_sweep per resample) against run_gibbs (graph replay in segments)
    m3, _ = _chain_model(use_graph=0)
    Ws = []
    for step in range(5 + 2 * 6):
        m3.resample(Y)
        if step >= 5 and (step - 5) % 2 == 0:
            Ws.append((m3.W.copy(), m3.V.copy()))
    assert np.array_equal(np.array([w for w, _ in Ws]), r1['W'])
    assert np.array_equal(np.array([v for _, v in Ws]), r1['V'])


def test_checkpoint_resumes_bit_for_bit(tmp_path):
    m, Y = _chain_model()
    for _ in range(3):
        m.resample(Y)
    path = str(tmp_path / 'ck.npz')
    m.save_checkpoint(path)
    ra = m.run_gibbs(Y, nburn=2, nthin=1, nsamples=3, verbose=False)
    m2, _ = _chain_model()
    m2._upload(Y)
    m2.load_checkpoint(path)
    rb = m2.run_gibbs(Y, nburn=2, nthin=1, nsamples=3, verbose=False)
    assert np.array_equal(ra['W'], rb['W']) and np.array_equal(ra['V'], rb['V'])


def test_evaluator_poisson_loglik_and_track_mu(tmp_path):
    from functionalmf_b200 import HeldOutEvaluator
    m, Y = _chain_model()
    ev = HeldOutEvaluator(m, Y, loglik='poisson')
    res = m.run_gibbs(Y, nburn=3, nthin=1, nsamples=4, verbose=False, track_mu=True, results_dir=str(tmp_path))
    Mu = np.einsum('znk,zmtk->znmt', res['W'], res['V'])
    obs = ~np.isnan(Y)
    with np.errstate(all='ignore'):
        ll = np.array([poisson.logpmf(Y[obs], mu[obs]).sum() / obs.sum() for mu in Mu])
    assert abs(ev.loglik()['all'] - ll.mean()) < 1e-10
    assert np.allclose(res['Mu_mean'], Mu.mean(axis=0), rtol=1e-12, atol=1e-12)
    assert os.path.exists(os.path.join(str(tmp_path), 'W.npy'))
    assert np.isfinite(m.logprob(Y))


def test_callback_keeps_the_per_sweep_loop():
    m, Y = _chain_model()
    seen = []
    res = m.run_gibbs(Y, nburn=1, nthin=1, nsamples=2, verbose=False, callback=lambda mm, d, s, **k: seen.append(s))
    assert seen == [0, 1, 2] and res['W'].shape == (2,) + m.W.shape


# ------------------------------------------------------------------ 4. refusals
def test_refusals():
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    from functionalmf_b200 import NonconjugateBayesianTensorFiltering
    from functionalmf_b200 import _lib as L
    from functionalmf_b200.engine import Engine
    m, Y = _chain_model()
    # invalid start: nothing changes
    W_bad = m.W.copy()
    W_bad[2, 0] = -5.0
    m.W = W_bad.copy()
    V0 = m.V.copy()
    with pytest.raises(L.BTFError) as ex:
        m.resample(Y)
    assert ex.value.code == L.BTF_ESTATE and 'row' in str(ex.value)
    assert np.array_equal(m._engine.get('W'), W_bad) and np.array_equal(m._engine.get('V'), V0)
    # counts that are not non-negative integers
    m2, _ = _chain_model()
    Yb = Y.copy()
    Yb[0, 0, 0], Yb[1, 1, 1] = -1.0, 1.5
    with pytest.raises(L.BTFError) as ex:
        m2.resample(Yb)
    assert ex.value.code == L.BTF_EINVAL and '2 observed' in str(ex.value)
    # EP with NaN
    N, M, T = m.nrows, m.ncols, m.ndepth
    mu, sg = np.ones((N, M, T)), np.ones((N, M, T))
    mu[0, 0, 0] = np.nan
    with pytest.raises(L.BTFError) as ex:
        m2._engine.set_ep(mu, sg)
    assert ex.value.code == L.BTF_EINVAL and '1 cell' in str(ex.value)
    # grids and shapes
    eng = m2._engine
    A, C = np.eye(T), np.zeros(T)
    g = np.linspace(-np.pi, np.pi, 100)
    with pytest.raises(L.BTFError):
        eng.set_gass(A, C, g, np.linspace(-np.pi, np.pi, 101))          # ngrid > ngrid_fine
    with pytest.raises(L.BTFError):
        eng.set_gass(A, C, g[::-1], g[:10])                              # fine grid not ascending
    with pytest.raises(ValueError):
        eng.set_gass(A, C[:-1], g, g[:10])
    with pytest.raises(L.BTFError):
        CM(N, M, T, 'poisson', np.zeros((0, T + 1)), nembeds=3, tf_order=1, gass_ngrid=0, seed=1).resample(Y)
    with pytest.raises(ValueError):
        CM(N, M, T, 'gaussian', np.zeros((0, T + 1)), nembeds=3, seed=1)
    with pytest.raises(ValueError):
        NonconjugateBayesianTensorFiltering(N, M, T, 'poisson', nembeds=3, seed=1)
    # sharded engines
    with pytest.raises(L.BTFError) as ex:
        Engine(N, M, T, nembeds=3, tf_order=1, likelihood=L.POISSON, world_size=2, rank=0, row_begin=0, row_end=4,
               col_begin=0, col_end=2)
    assert ex.value.code == L.BTF_EINVAL


# ------------------------------------------------------------------ 5. posterior against the host callable path
def test_posterior_matches_host_path():
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    rs = np.random.RandomState(8)
    N, M, T, K = 4, 3, 6, 2
    Wt = np.abs(rs.normal(size=(N, K))) + 0.5; Wt[np.triu_indices(K, k=1)] = 0
    Vt = np.abs(rs.normal(size=(M, T, K))) + 0.5
    Y = rs.poisson(np.einsum('nk,mtk->nmt', Wt, Vt) * 3).astype(float)
    cons = np.concatenate([np.eye(T), np.zeros((T, 1))], axis=1)
    nburn, nsamples, nbatch, nchains = 100, 400, 20, 2
    summaries = []
    for ll in (rowcol_loglikelihood, 'poisson'):
        m1 = np.zeros((nchains, nbatch, N, M, T))
        for c in range(nchains):
            np.random.seed(100 + c)
            m = CM(N, M, T, ll, cons, nembeds=K, tf_order=1, gass_ngrid=30, W_init=Wt, V_init=Vt * 3, seed=200 + c)
            res = m.run_gibbs(Y, nburn=nburn, nthin=1, nsamples=nsamples, verbose=False)
            Mu = np.einsum('znk,zmtk->znmt', res['W'], res['V'])
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
