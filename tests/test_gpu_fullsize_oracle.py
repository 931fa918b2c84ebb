"""Oracle parity AT the BASELINE shapes (VERDICT r1, missing #6).

The headline numbers come from code paths that small tensors never reach (the no-split two-CTA int8 GEMM, 128-row
linear-block tiles, one-wave splits, the look-ahead band kernel at full column counts).  These tests run ONE sweep
of the engine at the full configuration with injected noise and compare, for a sample of rows and of columns, every
stage with oracle/btf_oracle.py (the CPU restatement pinned to the reference fixtures): sufficient statistics,
row precision / factor / draw, assembled band, conditional mean and draw.  The oracle only ever sees the sampled
rows (all columns) and the sampled columns (all rows), so it finishes in seconds.

Tolerances: 1e-10 normwise for statistics / bands / row systems (north_star (a)); V means and draws
max(1e-10, 50 kappa eps) plus a 1e-13 backward error, exactly as tests/test_gpu_parity.py.
"""
import numpy as np
import pytest

from golden_util import normerr, relerr
from gpu_util import band_rows_from_lower

pytestmark = pytest.mark.gpu
TOL = 1e-10
EPS = np.finfo(float).eps


def _run_case(N, M, T, R, K, order, rows_s, cols_s, piece=256, seed=5, expect_i8=True):
    import torch
    from oracle import btf_oracle as O
    from functionalmf_b200.engine import Engine
    dev = torch.device('cuda', 0)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    rs = np.random.RandomState(seed)
    rows_s, cols_s = np.asarray(sorted(rows_s)), np.asarray(sorted(cols_s))
    eng = Engine(N, M, T, nembeds=K, tf_order=order, seed=11)
    Delta = eng.get('Delta')
    RD = Delta.shape[0]
    V0 = (torch.randn(M, T, K, generator=g, device=dev, dtype=torch.float64) * 0.3).cumsum(1)
    Yrows = np.empty((len(rows_s), M, T, R))
    Ycols = np.empty((N, len(cols_s), T, R))
    cols_t = torch.from_numpy(cols_s).to(dev)
    for a in range(0, N, piece):
        b = min(N, a + piece)
        Wg = torch.randn(b - a, K, generator=g, device=dev, dtype=torch.float64)
        Y = (Wg @ V0.reshape(M * T, K).T).reshape(b - a, M, T, 1) + \
            torch.randn(b - a, M, T, R, generator=g, device=dev, dtype=torch.float64)
        Y[torch.rand(Y.shape, generator=g, device=dev) < 0.2] = float('nan')
        torch.cuda.synchronize()
        eng.set_data_gaussian_rows_device(Y.data_ptr(), a, b - a, R, a == 0)
        Ycols[a:b] = Y[:, cols_t].cpu().numpy()
        for q, i in enumerate(rows_s):
            if a <= i < b:
                Yrows[q] = Y[i - a].cpu().numpy()
        del Y, Wg
    # state and noise of this sweep (W, V steps only: the hyper-parameter steps are covered at every shape by
    # tests/test_gpu_parity.py and do not depend on the tensor size)
    W0 = rs.normal(size=(N, K))
    W0[np.triu_indices(min(N, K), k=1, m=K)] = 0
    V0h = V0.cpu().numpy() + 0.05 * rs.normal(size=(M, T, K))
    Tau2 = rs.gamma(2.0, 1.0, size=(M, RD)) + 0.05
    sc = dict(lam2=0.7, lam2_a=1.3, sigma2=0.9, nu2=1.1)
    zW, zV = rs.normal(size=(N, K)), rs.normal(size=(M, T, K))
    eng.set('W', W0); eng.set('V', V0h)
    for nm in ('Tau2', 'Tau2_a', 'Tau2_b', 'Tau2_c'):
        eng.set(nm, Tau2)
    for k, v in sc.items():
        eng.set(k, [v])
    eng.set_sample_mask(16 | 32)
    eng.enable_diag(True)
    eng.inject('z_W', zW); eng.inject('z_V', zV)
    eng.sweep(1)
    Lp = K * (K + 1) // 2
    il = np.tril_indices(K)

    # ---- W step on the sampled rows
    cnt_r, S_r, _ = O.prereduce(Yrows)
    cw, sw = O.gaussian_weights(cnt_r, S_r, sc['nu2'])
    A, b_ = O.row_stats(V0h, cnt_r.astype(float), S_r)
    rstat = eng.diag('row_stats')[rows_s]
    assert normerr(rstat[:, :Lp], A[:, il[0], il[1]]) < TOL
    assert normerr(rstat[:, Lp:], b_) < TOL
    # element-wise on the diagonal of the product block (sums of non-negative terms: no cancellation)
    dg = [k * (k + 1) // 2 + k for k in range(K)]
    assert np.max(np.abs(rstat[:, dg] / A[:, range(K), range(K)] - 1.0)) < TOL
    Wn_s, dW = O.step_W(W0[rows_s], V0h, cw, sw, sc['sigma2'], zW[rows_s], row_index=rows_s)
    Wq = eng.diag('W_Q')[rows_s]
    Wl = eng.diag('W_L')[rows_s]
    Wg_all = eng.get('W')
    for q, i in enumerate(rows_s):
        d = min(i + 1, K)
        assert normerr(Wq[q][:d, :d], dW['Q'][q][:d, :d]) < TOL, ('W_Q', i)
        assert normerr(np.tril(Wl[q][:d, :d]), dW['L'][q][:d, :d]) < 1e-9, ('W_L', i)
    assert normerr(Wg_all[rows_s], Wn_s) < 1e-9
    assert np.all(Wg_all[np.triu_indices(min(N, K), k=1, m=K)] == 0)

    # ---- V step on the sampled columns, given the engine's new W (checked above on the row sample)
    cnt_c, S_c, _ = O.prereduce(Ycols)
    Ac, bc = O.col_stats(Wg_all, cnt_c.astype(float), S_c)
    cstat = eng.diag('col_stats').reshape(M, T, Lp + K)[cols_s]
    assert normerr(cstat[..., :Lp], Ac[..., il[0], il[1]]) < TOL
    assert normerr(cstat[..., Lp:], bc) < TOL
    assert np.max(np.abs(cstat[..., dg] / Ac[..., range(K), range(K)] - 1.0)) < TOL
    cwc, swc = O.gaussian_weights(cnt_c, S_c, sc['nu2'])
    Vn, dV = O.step_V(Wg_all, V0h[cols_s], cwc, swc, Delta, sc['lam2'], Tau2[cols_s], zV[cols_s], order, want_diag=True)
    band = eng.diag('V_band')[cols_s]
    mean = eng.diag('V_mean')[cols_s]
    Vg = eng.get('V')
    assert int(eng.diag('V_retries').sum()) == 0 and int(dV['retries'].sum()) == 0
    for q, j in enumerate(cols_s):
        assert normerr(band[q], band_rows_from_lower(dV['band'][q])) < TOL, ('band', j)
        Qd = O.band_to_dense_lower(dV['band'][q])
        Qd = Qd + np.tril(Qd, -1).T
        kappa = np.linalg.cond(Qd)
        tol = max(TOL, 50 * kappa * EPS)
        assert normerr(mean[q], dV['mean'][q]) < tol, ('mean', j, kappa)
        assert normerr(Vg[j], Vn[q]) < tol, ('draw', j, kappa)
        rhs = dV['b'][q].ravel()
        m = mean[q].ravel()
        bwd = np.linalg.norm(Qd @ m - rhs) / (np.linalg.norm(Qd, 2) * np.linalg.norm(m) + np.linalg.norm(rhs))
        assert bwd < 1e-13, (j, bwd)
    # the headline configuration must be on the integer-tensor-core path (and this test must say so if not)
    ph = eng.time_phases(1)
    assert (ph.get('row_i8gemm', 0.0) > 0.0) == expect_i8
    eng.close()


def test_c2_shape_sampled_rows_and_columns_vs_oracle():
    """BASELINE.json configs[1]: 4096 x 1024 x 64 x 3, nembeds=16, tf_order=2, 20 % NaN; 16 rows, 2 columns."""
    rs = np.random.RandomState(1)
    rows = [0, 3, 15, 16] + sorted(rs.choice(np.arange(17, 4096), 12, replace=False).tolist())
    _run_case(4096, 1024, 64, 3, 16, 2, rows, [0, 777])


def test_c5_slice_k32_sampled_rows_and_columns_vs_oracle():
    """A slice of BASELINE.json configs[4] (65536 x 8192 x 128 x 2, nembeds=32): same depth, replicates, embedding
    size and per-column system (n = 4096, half-bandwidth 96) with 2048 rows and 1024 columns, so that the diagnostic
    copies of the bands fit next to the data; 8 rows, 2 columns."""
    rs = np.random.RandomState(2)
    rows = [0, 31, 32] + sorted(rs.choice(np.arange(33, 2048), 5, replace=False).tolist())
    _run_case(2048, 1024, 128, 2, 32, 2, rows, [5, 1023], piece=128)


def test_c3_shape_binomial_sampled_rows_and_columns_vs_oracle():
    """BASELINE.json C3 (Binomial, 4096 x 1024 x 32, 4 trials, 1 % NaN, nembeds=8, tf_order=1): one W, V sweep with
    injected Polya-Gamma weights through the f64-weight statistics kernels at full size; 16 rows, 2 columns.  The
    weights are real, so the integer-tensor-core path must stay off."""
    from oracle import btf_oracle as O
    from functionalmf_b200.engine import Engine
    N, M, T, K, order, trials = 4096, 1024, 32, 8, 1, 4
    rs = np.random.RandomState(3)
    rows_s = np.asarray([0, 7, 31, 32] + sorted(rs.choice(np.arange(33, N), 12, replace=False).tolist()))
    cols_s = np.asarray([1, 1023])
    W0 = rs.normal(size=(N, K))
    W0[np.triu_indices(K, k=1)] = 0
    V0 = rs.normal(size=(M, T, K)).cumsum(axis=1) * 0.2
    # data, trials and weights in 256-row pieces (three 1 GB host arrays, no full-size temporaries)
    Ys = np.empty((N, M, T))
    Nt = np.empty((N, M, T))
    omega = np.empty((N, M, T))
    Vf = V0.reshape(M * T, K)
    for a in range(0, N, 256):
        b = min(N, a + 256)
        mu = (W0[a:b] @ Vf.T).reshape(b - a, M, T) * 0.5
        y = rs.binomial(trials, 1 / (1 + np.exp(-mu))).astype(float)
        miss = rs.random_sample(y.shape) < 0.01
        y[miss] = np.nan
        Ys[a:b] = y
        Nt[a:b] = np.where(miss, np.nan, float(trials))
        omega[a:b] = np.where(miss, 0.0, rs.gamma(2.0, 0.2, size=y.shape) + 0.02)
    eng = Engine(N, M, T, nembeds=K, tf_order=order, likelihood=1, seed=11)
    Delta = eng.get('Delta')
    RD = Delta.shape[0]
    eng.set_data_binomial(Ys, Nt)
    Wst = W0 + 0.05 * rs.normal(size=(N, K)) * (W0 != 0)
    Vst = V0 + 0.05 * rs.normal(size=(M, T, K))
    Tau2 = rs.gamma(2.0, 1.0, size=(M, RD)) + 0.05
    sc = dict(lam2=0.7, lam2_a=1.3, sigma2=0.9)
    zW, zV = rs.normal(size=(N, K)), rs.normal(size=(M, T, K))
    eng.set('W', Wst); eng.set('V', Vst)
    for nm in ('Tau2', 'Tau2_a', 'Tau2_b', 'Tau2_c'):
        eng.set(nm, Tau2)
    for k, v in sc.items():
        eng.set(k, [v])
    eng.set_sample_mask(16 | 32)
    eng.enable_diag(True)
    eng.inject('omega', omega)
    eng.inject('z_W', zW); eng.inject('z_V', zV)
    eng.sweep(1)
    Lp = K * (K + 1) // 2
    il = np.tril_indices(K)
    dg = [k * (k + 1) // 2 + k for k in range(K)]

    # ---- W step on the sampled rows
    cw, sw = O.binomial_weights(Ys[rows_s], Nt[rows_s], omega[rows_s])
    A, b_ = O.row_stats(Vst, cw, sw)
    rstat = eng.diag('row_stats')[rows_s]
    assert normerr(rstat[:, :Lp], A[:, il[0], il[1]]) < TOL
    assert normerr(rstat[:, Lp:], b_) < TOL
    assert np.max(np.abs(rstat[:, dg] / A[:, range(K), range(K)] - 1.0)) < TOL
    Wn_s, dW = O.step_W(Wst[rows_s], Vst, cw, sw, sc['sigma2'], zW[rows_s], row_index=rows_s)
    Wq = eng.diag('W_Q')[rows_s]
    Wl = eng.diag('W_L')[rows_s]
    Wg_all = eng.get('W')
    for q, i in enumerate(rows_s):
        d = min(i + 1, K)
        assert normerr(Wq[q][:d, :d], dW['Q'][q][:d, :d]) < TOL, ('W_Q', i)
        assert normerr(np.tril(Wl[q][:d, :d]), dW['L'][q][:d, :d]) < 1e-9, ('W_L', i)
    assert normerr(Wg_all[rows_s], Wn_s) < 1e-9
    assert np.all(Wg_all[np.triu_indices(K, k=1)] == 0)

    # ---- V step on the sampled columns, given the engine's new W
    cwc, swc = O.binomial_weights(Ys[:, cols_s], Nt[:, cols_s], omega[:, cols_s])
    del Ys, Nt, omega
    Ac, bc = O.col_stats(Wg_all, cwc, swc)
    cstat = eng.diag('col_stats').reshape(M, T, Lp + K)[cols_s]
    assert normerr(cstat[..., :Lp], Ac[..., il[0], il[1]]) < TOL
    assert normerr(cstat[..., Lp:], bc) < TOL
    assert np.max(np.abs(cstat[..., dg] / Ac[..., range(K), range(K)] - 1.0)) < TOL
    Vn, dV = O.step_V(Wg_all, Vst[cols_s], cwc, swc, Delta, sc['lam2'], Tau2[cols_s], zV[cols_s], order, want_diag=True)
    band = eng.diag('V_band')[cols_s]
    mean = eng.diag('V_mean')[cols_s]
    Vg = eng.get('V')
    assert int(eng.diag('V_retries').sum()) == 0 and int(dV['retries'].sum()) == 0
    for q, j in enumerate(cols_s):
        assert normerr(band[q], band_rows_from_lower(dV['band'][q])) < TOL, ('band', j)
        Qd = O.band_to_dense_lower(dV['band'][q])
        Qd = Qd + np.tril(Qd, -1).T
        kappa = np.linalg.cond(Qd)
        tol = max(TOL, 50 * kappa * EPS)
        assert normerr(mean[q], dV['mean'][q]) < tol, ('mean', j, kappa)
        assert normerr(Vg[j], Vn[q]) < tol, ('draw', j, kappa)
        rhs = dV['b'][q].ravel()
        m = mean[q].ravel()
        bwd = np.linalg.norm(Qd @ m - rhs) / (np.linalg.norm(Qd, 2) * np.linalg.norm(m) + np.linalg.norm(rhs))
        assert bwd < 1e-13, (j, bwd)
    ph = eng.time_phases(1)
    assert ph.get('row_i8gemm', 0.0) == 0.0
    eng.close()
