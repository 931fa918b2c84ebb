"""The negative-binomial dispersion (R) step against oracle.btf_oracle.step_R, on both of its device routes.

launch_nb_update (pg_kernels.cu) runs the random-walk Metropolis chain of R in one of two ways:
  * histogram route (nb_mh_hist_kernel): integer counts with (max count + 1) * groups <= 2^24; the sum of
    lgamma(y + r) over a group is taken from a per-group count histogram, the whole chain in one block;
  * direct route (nb_mh_kernel + nb_lgamma_kernel): any other data, or BTF_NB_NO_HIST set when the engine is created;
    per step a pass over the data with warp-aggregated atomics.
The proposal normals and acceptance uniforms are injected, so device and oracle make the same decisions.  The
oracle also reports how close its nearest decision came to a tie (|u - prob| / prob); noise with a margin below
1e-6 is redrawn, so a disagreement is a bug and not a rounding tie.  Which route ran is read from the engine's
launch counter: building the histogram adds 2 launches to set_data_negbin; the R update adds 4 launches on the
histogram route and 2 nmh + 4 on the direct route, against 1 (pseudo-counts only) without it.
"""
import numpy as np
import pytest

from functionalmf_b200._lib import NEGBINOMIAL, SAMPLE_R
from golden_util import normerr, relerr
from gpu_util import band_rows_from_lower

pytestmark = pytest.mark.gpu
RPROP, RSTD = 0.2, 1.0
MARGIN = 1e-6


def _counts(rs, W, V, nreps, nan_frac, scale=1.0):
    """Counts generated as in tools/bench_configs.py (c4): Poisson(Gamma(5, P / (1 - P))), P = ilogit(mu)."""
    Mu = np.einsum('nk,mtk->nmt', W, V)
    Mu = 2 * Mu / np.abs(Mu).max()
    P = 1 / (1 + np.exp(-Mu))
    lam = rs.gamma(5.0, scale * P / (1 - P), size=(nreps,) + Mu.shape)
    Y = np.moveaxis(rs.poisson(lam).astype(float), 0, -1)
    Y[rs.random_sample(Y.shape) < nan_frac] = np.nan
    return Y


def _r_shape(mask, N, M, T):
    return tuple(1 if mask >> d & 1 else s for d, s in enumerate((N, M, T)))


def _noise_with_margin(R0, W, V, Y, mask, nmh, seed):
    """Oracle chain for injected noise whose closest accept/reject decision is > MARGIN away from a tie."""
    from oracle import btf_oracle as O
    rdims = [d for d in range(3) if mask >> d & 1]
    for k in range(20):
        rr = np.random.RandomState(seed + k)
        zs = rr.normal(size=(nmh,) + R0.shape)
        us = rr.random_sample((nmh,) + R0.shape)
        Rw, Nw, margin = O.step_R(R0, W, V, Y, rdims, zs, us, RPROP, RSTD, want_margin=True)
        if margin > MARGIN:
            return zs, us, Rw, Nw
    raise AssertionError('no noise draw without a near-tie in 20 seeds')


def _run_r_step(Y, W, V, R0, mask, nmh, zs, us, seed=1):
    """One sweep with the sample mask set to R alone; returns (engine, histogram built, launches of the R update)."""
    from functionalmf_b200.engine import Engine
    N, M, T = Y.shape[:3]
    eng = Engine(N, M, T, nembeds=W.shape[1], tf_order=2, likelihood=NEGBINOMIAL, seed=seed, use_graph=0,
                 nmetropolis=nmh, rpropstdev=RPROP, rstdev=RSTD, rdims_mask=mask)
    l0 = eng.kernel_launches
    eng.set_data_negbin(Y)
    hist = eng.kernel_launches - l0
    assert hist in (0, 2)
    eng.set('W', W)
    eng.set('V', V)
    eng.set('R', R0)
    eng.set_sample_mask(0)                 # pseudo-counts only: the launch count without the R update
    l0 = eng.kernel_launches
    eng.sweep(1)
    base = eng.kernel_launches - l0
    if nmh:
        eng.inject('z_R', zs)
        eng.inject('u_R', us)
    eng.set_sample_mask(SAMPLE_R)
    l0 = eng.kernel_launches
    eng.sweep(1)
    extra = eng.kernel_launches - l0 - base + 1
    return eng, hist == 2, extra


def _check_route(hist, extra, nmh, want_hist):
    assert hist == want_hist
    if nmh:
        assert extra == (4 if want_hist else 2 * nmh + 4), (hist, extra)
    else:
        assert extra == 1


def _check_against_oracle(eng, Y, R0, Rw, Nw, nmh):
    obs = np.any(~np.isnan(Y), axis=-1)
    Rg = eng.get('R')
    assert relerr(Rg, Rw) < 1e-12
    if nmh:
        assert np.any(Rw != R0)                # the chain moved: the comparison is not of untouched inputs
    Ng, kap = eng.get('Ntrials'), eng.get('kappa')
    assert np.max(np.abs(Ng[obs] / Nw[obs] - 1.0)) < 1e-12
    kref = np.nansum(Y, axis=-1) - Nw / 2
    assert np.max(np.abs(kap[obs] - kref[obs]) / Nw[obs]) < 1e-12
    assert np.all(Ng[~obs] == 0.0) and np.all(kap[~obs] == 0.0)


@pytest.mark.parametrize('nmh', [0, 30, 300])
@pytest.mark.parametrize('route', ['hist', 'direct'])
@pytest.mark.parametrize('mask', range(8))
def test_r_step_matrix(mask, route, nmh, monkeypatch):
    """All eight rdims layouts x both routes x nmh in {0, 30, 300} (300 > 256: the histogram kernel draws its noise
    inside the loop instead of up front), 40 x 7 x 13 x 2 integer counts, 15 % missing."""
    N, M, T, R, K = 40, 7, 13, 2, 3
    rs = np.random.RandomState(100 + mask)
    W = rs.normal(size=(N, K))
    V = rs.normal(size=(M, T, K)).cumsum(axis=1) * 0.3
    Y = _counts(rs, W, V, R, 0.15)
    Y[0, 0, 0, :] = np.nan                 # one cell with no observation at all
    R0 = rs.uniform(1.5, 8.0, size=_r_shape(mask, N, M, T))
    zs, us, Rw, Nw = _noise_with_margin(R0, W, V, Y, mask, nmh, 1000 * mask + nmh)
    if route == 'direct':
        monkeypatch.setenv('BTF_NB_NO_HIST', '1')
    else:
        monkeypatch.delenv('BTF_NB_NO_HIST', raising=False)
    eng, hist, extra = _run_r_step(Y, W, V, R0, mask, nmh, zs, us)
    _check_route(hist, extra, nmh, route == 'hist')
    _check_against_oracle(eng, Y, R0, Rw, Nw, nmh)
    eng.close()


@pytest.mark.parametrize('mask', [0, 5, 7])
def test_r_step_non_integer_counts_take_direct_route(mask, monkeypatch):
    monkeypatch.delenv('BTF_NB_NO_HIST', raising=False)
    N, M, T, R, K, nmh = 40, 7, 13, 2, 3, 30
    rs = np.random.RandomState(7 + mask)
    W = rs.normal(size=(N, K))
    V = rs.normal(size=(M, T, K)).cumsum(axis=1) * 0.3
    Y = _counts(rs, W, V, R, 0.15)
    Y[rs.random_sample(Y.shape) < 0.2] += 0.5
    R0 = rs.uniform(1.5, 8.0, size=_r_shape(mask, N, M, T))
    zs, us, Rw, Nw = _noise_with_margin(R0, W, V, Y, mask, nmh, 77 + mask)
    eng, hist, extra = _run_r_step(Y, W, V, R0, mask, nmh, zs, us)
    _check_route(hist, extra, nmh, False)
    _check_against_oracle(eng, Y, R0, Rw, Nw, nmh)
    eng.close()


def test_r_step_per_cell_wide_count_range_takes_direct_route(monkeypatch):
    """rdims = () at 60 x 30 x 40: 72 000 groups x (300 + 1) histogram bins > 2^24, so the direct route runs."""
    monkeypatch.delenv('BTF_NB_NO_HIST', raising=False)
    N, M, T, R, K, nmh = 60, 30, 40, 1, 4, 30
    rs = np.random.RandomState(11)
    W = rs.normal(size=(N, K))
    V = rs.normal(size=(M, T, K)).cumsum(axis=1) * 0.3
    Y = _counts(rs, W, V, R, 0.1)
    Y[rs.random_sample(Y.shape) < 0.01] = 300.0
    assert (np.nanmax(Y) + 1) * N * M * T > (1 << 24)
    R0 = rs.uniform(1.5, 8.0, size=(N, M, T))
    zs, us, Rw, Nw = _noise_with_margin(R0, W, V, Y, 0, nmh, 5)
    eng, hist, extra = _run_r_step(Y, W, V, R0, 0, nmh, zs, us)
    _check_route(hist, extra, nmh, False)
    _check_against_oracle(eng, Y, R0, Rw, Nw, nmh)
    eng.close()


@pytest.mark.parametrize('mask', [7, 0])
def test_c4_shape_whole_sweep_vs_oracle(mask, monkeypatch):
    """BASELINE C4 (19 x 19 x 228, K = 10, tf_order 2, 30 MH steps), rdims (0,1,2) and (): one whole negative-binomial
    sweep with injected noise (R chain, omega, sigma2, Tau2, lam2, W, V) against the oracle on all rows and columns.
    19 band systems of 228 block rows (half-bandwidth 30), K = 10 padded to 16 in the device kernels."""
    from oracle import btf_oracle as O
    from functionalmf_b200.engine import Engine
    from scipy.linalg import eigvals_banded
    monkeypatch.delenv('BTF_NB_NO_HIST', raising=False)
    N, M, T, K, order, nmh = 19, 19, 228, 10, 2, 30
    rs = np.random.RandomState(40 + mask)
    W = rs.normal(size=(N, K))
    W[np.triu_indices(K, k=1)] = 0
    V = (rs.normal(size=(M, T, K)) * (rs.random_sample((M, T, 1)) < 0.3)).cumsum(axis=1) * 0.5
    Y = _counts(rs, W, V, 1, 0.1025)
    eng = Engine(N, M, T, nembeds=K, tf_order=order, likelihood=NEGBINOMIAL, seed=3, use_graph=0,
                 nmetropolis=nmh, rpropstdev=RPROP, rstdev=RSTD, rdims_mask=mask)
    Delta = eng.get('Delta')
    RD = Delta.shape[0]
    st = dict(W=W + 0.05 * rs.normal(size=W.shape) * (W != 0), V=V + 0.05 * rs.normal(size=V.shape),
              Tau2=rs.gamma(2.0, 1.0, size=(M, RD)) + 0.05, Tau2_a=rs.gamma(2.0, 1.0, size=(M, RD)) + 0.05,
              Tau2_b=rs.gamma(2.0, 1.0, size=(M, RD)) + 0.05, Tau2_c=rs.gamma(2.0, 1.0, size=(M, RD)) + 0.05,
              lam2=0.7, lam2_a=1.3, sigma2=0.9)
    R0 = rs.uniform(1.5, 8.0, size=_r_shape(mask, N, M, T))
    zs, us, Rw, Nw = _noise_with_margin(R0, st['W'], st['V'], Y, mask, nmh, 300 + mask)
    obs = np.any(~np.isnan(Y), axis=-1)
    noise = dict(g_sigma2=rs.gamma(20.0), g_tau=rs.gamma(2.0, size=(M, 4, RD)) + 1e-3, g_lam=rs.gamma(30.0, size=2),
                 z_W=rs.normal(size=(N, K)), z_V=rs.normal(size=(M, T, K)),
                 omega=np.where(obs, rs.gamma(2.0, 0.15, size=(N, M, T)) + 0.02, 0.0))
    # the PG step of a negative-binomial sweep sees Binomial pseudo-data: successes sum_obs y, trials sum_obs (y + R)
    Ysum = np.where(obs, np.nansum(Y, axis=-1), np.nan)
    Ntr = np.where(obs, Nw, np.nan)
    cfg = dict(K=K, order=order, Delta=Delta, sigma2_a=0.1, sigma2_b=0.1, stability=1e-6, force_psd=True,
               force_psd_eps=1e-6, force_psd_attempts=4, ref_compat=True)
    want = O.binomial_sweep(st, Ysum, Ntr, noise, cfg)

    eng.set_data_negbin(Y)
    eng.enable_diag(True)
    for k in ('W', 'V', 'Tau2', 'Tau2_a', 'Tau2_b', 'Tau2_c'):
        eng.set(k, st[k])
    for k in ('lam2', 'lam2_a', 'sigma2'):
        eng.set(k, [st[k]])
    eng.set('R', R0)
    for k, v in noise.items():
        eng.inject(k, np.atleast_1d(v))
    eng.inject('z_R', zs)
    eng.inject('u_R', us)
    eng.sweep(1)

    _check_against_oracle(eng, Y, R0, Rw, Nw, nmh)
    for k in ('sigma2', 'lam2', 'lam2_a'):
        assert relerr(eng.get_scalar(k), want[k]) < 1e-10, k
    for k in ('Tau2', 'Tau2_a', 'Tau2_b', 'Tau2_c'):
        assert relerr(eng.get(k), want[k]) < 1e-10, k
    cw, sw = O.binomial_weights(Ysum, Ntr, noise['omega'])
    Lp = K * (K + 1) // 2
    il = np.tril_indices(K)
    A, b = O.row_stats(st['V'], cw, sw)
    rstat = eng.diag('row_stats')
    assert normerr(rstat[:, :Lp], A[:, il[0], il[1]]) < 1e-10
    assert normerr(rstat[:, Lp:], b) < 1e-10
    Ac, bc = O.col_stats(want['W'], cw, sw)
    cstat = eng.diag('col_stats')
    assert normerr(cstat[:, :Lp], Ac.reshape(M * T, K, K)[:, il[0], il[1]]) < 1e-10
    assert normerr(cstat[:, Lp:], bc.reshape(M * T, K)) < 1e-10
    assert normerr(eng.get('W'), want['W']) < 1e-9
    Vn, dV = O.step_V(want['W'], st['V'], cw, sw, Delta, want['lam2'], want['Tau2'], noise['z_V'], order,
                      want_diag=True)
    band, mean, Vg = eng.diag('V_band'), eng.diag('V_mean'), eng.get('V')
    eps = np.finfo(float).eps
    for j in range(M):
        assert normerr(band[j], band_rows_from_lower(dV['band'][j])) < 1e-10, ('band', j)
        ev = eigvals_banded(dV['band'][j], lower=True)
        kappa = ev.max() / ev.min()
        tol = max(1e-10, 50 * kappa * eps)
        assert normerr(mean[j], dV['mean'][j]) < tol, ('mean', j, kappa)
        assert normerr(Vg[j], Vn[j]) < tol, ('draw', j, kappa)
        Qd = O.band_to_dense_lower(dV['band'][j])
        Qd = Qd + np.tril(Qd, -1).T
        rhs, m = dV['b'][j].ravel(), mean[j].ravel()
        bwd = np.linalg.norm(Qd @ m - rhs) / (ev.max() * np.linalg.norm(m) + np.linalg.norm(rhs))
        assert bwd < 1e-13, (j, bwd)
    eng.close()
