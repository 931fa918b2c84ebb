"""CPU restatement (numpy/scipy) of the BTF Gibbs sweep.  TEST INFRASTRUCTURE ONLY.

This is the parity oracle for the CUDA engine: every conditional of one
``resample(data)`` call of the reference, written as a pure function of the
current state, the data and an explicit *noise* record (standard normal /
standard gamma / uniform / Polya-Gamma variates), so that the reference, this
oracle and the GPU engine can be driven with identical randomness.

Pinned against the reference itself: ``oracle/make_golden.py`` imports the
unmodified reference from /root/reference (with the import shims under
``oracle/shims``), records its noise and its state after every step, and
``tests/test_oracle_golden.py`` checks this file against those fixtures.
The reference has no tests or golden vectors of its own (SURVEY.md section 4).

Conventions
-----------
* ``V`` is ``[M, T, K]``; the V-conditional is solved in **t-major** order
  (``x[t*K + k] = V[j, t, k]``), i.e. the reference's k-major system
  (factor.py:189, 409) permuted by ``P[t*K+k] = k*T+t`` -- the permutation the
  sksparse shim reports, so ``z`` is consumed in the same order.
* Gamma noise is stored as *standard* variates ``g ~ Gamma(shape, 1)``;
  ``np.random.gamma(shape, scale)`` is ``g * scale``.
"""
import numpy as np
import scipy.linalg as sla


# ----------------------------------------------------------------------------
# trend-filtering penalty   (utils.py:56-98)
# ----------------------------------------------------------------------------
def first_difference(T):
    """(T-1) x T first-difference matrix, rows [-1, 1]  (utils.py:93-98)."""
    D = np.zeros((T - 1, T))
    i = np.arange(T - 1)
    D[i, i] = -1.0
    D[i, i + 1] = 1.0
    return D


def delta_matrix(T, order, anchor=0):
    """Dense Bayesian trend-filtering matrix (utils.py:56-90).

    Stack of the anchor row e_anchor^T and the difference operators of order
    0..``order`` where order k is obtained by alternately applying D^T and D
    (utils.py:61-64): D, D^T D, D D^T D, ...
    """
    D = first_difference(T)
    blocks = [np.zeros((1, T))]
    blocks[0][0, anchor] = 1.0
    for k in range(order + 1):
        cur = D
        for i in range(k):
            cur = D.T @ cur if i % 2 == 0 else D @ cur
        blocks.append(cur)
    return np.concatenate(blocks, axis=0)


# ----------------------------------------------------------------------------
# sufficient statistics of the data
# ----------------------------------------------------------------------------
def prereduce(Y):
    """Replicate pre-reduction (factor.py:323-330, 368-375).

    Returns ``cnt`` (# non-NaN replicates per cell), ``S`` (nansum over
    replicates) and the scalar total of squares over all observed entries.
    """
    Y = np.asarray(Y, dtype=float)
    if Y.ndim == 3:
        Y = Y[..., None]
    obs = ~np.isnan(Y)
    cnt = obs.sum(axis=-1)
    Y0 = np.where(obs, Y, 0.0)
    return cnt, Y0.sum(axis=-1), float((Y0 * Y0).sum())


def n_w_free(N, K):
    """Number of free entries of the lower-triangular W (factor.py:155-163)."""
    if N >= K:
        return (K * K - K) // 2 + K + (N - K) * K
    return (N * N - N) // 2 + N


def w_free_mask(N, K):
    m = np.ones((N, K), dtype=bool)
    d = min(N, K)
    iu = np.triu_indices(d, k=1, m=K)
    m[:d][iu] = False
    return m


# ----------------------------------------------------------------------------
# scalar / hyper-parameter conditionals
# ----------------------------------------------------------------------------
def inv_gamma_post(shape, rate, nobs, sqerr, g):
    """ConjugateInverseGammaPrior.resample (genlasso.py:149-168) -> variance."""
    a_post = shape + nobs / 2.0
    b_post = rate + sqerr / 2.0
    prec = g * (1.0 / b_post)
    return 1.0 / prec, a_post, b_post


def step_nu2(W, V, Y, nu2_a, nu2_b, g):
    """GaussianBTF._resample_nu2 (factor.py:411-416).  Returns (nu2, a, b)."""
    Y = np.asarray(Y, dtype=float)
    if Y.ndim == 3:
        Y = Y[..., None]
    Mu = np.einsum('nk,mtk->nmt', W, V)[..., None]
    obs = ~np.isnan(Y)
    sq = float((np.where(obs, Mu - np.where(obs, Y, 0.0), 0.0) ** 2).sum())
    return inv_gamma_post(nu2_a, nu2_b, int(obs.sum()), sq, g)


def step_sigma2(W, sigma2_a, sigma2_b, g):
    """BTF._resample_sigma2 (factor.py:130-132, 155-174)."""
    N, K = W.shape
    free = w_free_mask(N, K)
    sq = float((W[free] ** 2).sum())
    return inv_gamma_post(sigma2_a, sigma2_b, int(free.sum()), sq, g)


def step_tau2(V, Delta, lam2, Tau2_a, Tau2_b, Tau2_c, g, K, stability=1e-6):
    """BTF._resample_Tau2 (factor.py:134-141).  ``g`` is [M, 4, R_D] standard
    gammas in the order tau2 (shape (K+1)/2), c, b, a (shape 1)."""
    lo, hi = stability, 1.0 / stability
    deltas = np.einsum('rt,mtk->mrk', Delta, V)
    rate = (deltas ** 2).sum(axis=2) / (2 * lam2) + 1.0 / Tau2_c.clip(lo, hi)
    Tau2 = 1.0 / (g[:, 0] * (1.0 / rate.clip(lo, hi)))
    c = 1.0 / (g[:, 1] * (1.0 / (1.0 / Tau2 + 1.0 / Tau2_b).clip(lo, hi)))
    b = 1.0 / (g[:, 2] * (1.0 / (1.0 / c + 1.0 / Tau2_a).clip(lo, hi)))
    a = 1.0 / (g[:, 3] * (1.0 / (1.0 / b + 1.0).clip(lo, hi)))
    return Tau2, a, b, c


def step_lam2(V, Delta, Tau2, lam2_a, g, K, ref_compat=True):
    """BTF._resample_lam2 (factor.py:143-153).

    ``ref_compat=True`` reproduces the reference as written: the rate is
    *overwritten* for every column (factor.py:150), so only the last column
    contributes and the 1/lam2_a prior term is dropped.  ``False`` sums over
    all columns and keeps the prior term (the presumably intended update).
    """
    M = V.shape[0]
    deltas = np.einsum('rt,mtk->mrk', Delta, V)
    per_col = ((deltas / np.sqrt(Tau2)[:, :, None]) ** 2).sum(axis=(1, 2)) / 2.0
    rate = per_col[-1] if ref_compat else 1.0 / lam2_a + per_col.sum()
    shape = Delta.shape[0] * M * K + 1
    lam2 = max(1e-5, 1.0 / (g[0] * (1.0 / rate)))
    lam2_a_new = 1.0 / (g[1] * (1.0 / (1.0 / lam2 + 1.0)))
    return lam2, lam2_a_new, rate, shape / 2.0


# ----------------------------------------------------------------------------
# W step   (factor.py:313-362)
# ----------------------------------------------------------------------------
def row_stats(V, cw, sw):
    """Per-row statistics  A_i = sum_p cw[i,p] v_p v_p^T,  b_i = sum_p sw[i,p] v_p.

    ``cw`` is the precision weight (cnt/nu2 or omega) and ``sw`` the weighted
    sum (S/nu2 or y - n/2), both [N, M, T] and zero on missing cells.
    """
    K = V.shape[-1]
    Vf = V.reshape(-1, K)
    Z = (Vf[:, :, None] * Vf[:, None, :]).reshape(Vf.shape[0], K * K)
    N = cw.shape[0]
    A = (cw.reshape(N, -1) @ Z).reshape(N, K, K)
    b = sw.reshape(N, -1) @ Vf
    return A, b


def step_W(W, V, cw, sw, sigma2, z, row_index=None):
    """GaussianBTF._resample_W (factor.py:313-362) with explicit noise z [N, K].

    Returns (W_new, diag) where diag holds per-row Q (with the I/sigma2 prior,
    zero outside the leading d x d block), its lower Cholesky factor and the
    conditional mean.  ``row_index`` (optional) gives the position of every
    passed row in the full W (a sample of rows of a large problem): the first K
    rows are lower triangular, d = min(i + 1, K) with i the GLOBAL row index.
    """
    N, K = W.shape
    A, b = row_stats(V, cw, sw)
    Wn = W.copy()
    Qs = np.zeros((N, K, K))
    Ls = np.zeros((N, K, K))
    means = np.zeros((N, K))
    for i in range(N):
        d = min((i if row_index is None else int(row_index[i])) + 1, K)
        Q = A[i, :d, :d] + np.eye(d) / sigma2
        L = np.linalg.cholesky(Q)
        mean = sla.cho_solve((L, True), b[i, :d])
        Wn[i, :d] = mean + sla.solve_triangular(L.T, z[i, :d], lower=False)
        Qs[i, :d, :d], Ls[i, :d, :d], means[i, :d] = Q, L, mean
    return Wn, dict(Q=Qs, L=Ls, mean=means, b=b)


# ----------------------------------------------------------------------------
# V step   (factor.py:364-409, fast_mvn.py:10-74)
# ----------------------------------------------------------------------------
def col_stats(W, cw, sw):
    """Per-(column, depth) statistics A_jt = sum_i cw[i,j,t] w_i w_i^T [M,T,K,K]
    and b_jt = sum_i sw[i,j,t] w_i [M,T,K]  (factor.py:396-401 without kron)."""
    N, K = W.shape
    Z = (W[:, :, None] * W[:, None, :]).reshape(N, K * K)
    M, T = cw.shape[1], cw.shape[2]
    A = (cw.reshape(N, -1).T @ Z).reshape(M, T, K, K)
    b = (sw.reshape(N, -1).T @ W).reshape(M, T, K)
    return A, b


def prior_band(Delta, lam2, tau2_j):
    """T x T banded prior precision Delta^T diag(1/(lam2 tau2)) Delta (factor.py:404)."""
    return Delta.T @ ((1.0 / (lam2 * tau2_j))[:, None] * Delta)


def assemble_band(A_j, Pm, order):
    """Lower-banded (LAPACK 'ab', lower) storage of the t-major precision
    Q = blockdiag_t(A_jt) + Pm (x) I_K, half-bandwidth kd = (order+1) K."""
    T, K = A_j.shape[0], A_j.shape[1]
    n, kd = T * K, (order + 1) * K
    ab = np.zeros((kd + 1, n))
    for d in range(K):
        ab[d].reshape(T, K)[:, :K - d] = A_j[:, np.arange(d, K), np.arange(0, K - d)]
    for m in range(order + 2):
        if m < T:
            ab[m * K, :n - m * K] += np.repeat(np.diagonal(Pm, -m), K)
    return ab


def band_to_dense_lower(cb):
    kd, n = cb.shape[0] - 1, cb.shape[1]
    L = np.zeros((n, n))
    for d in range(kd + 1):
        idx = np.arange(n - d)
        L[idx + d, idx] = cb[d, :n - d]
    return L


def mvn_from_band(ab, rhs, z, force_psd=True, eps=1e-6, attempts=4):
    """sample_mvn_from_precision, sparse branch (fast_mvn.py:33-74), on a banded
    t-major system: x = Q^-1 rhs + L^-T z with jitter retry eps, 10 eps, ...

    Returns (x, mean, cb, n_retries).  Raises LinAlgError when the retries are
    exhausted (the reference would loop forever, SURVEY.md Q4)."""
    ab = ab.copy()
    attempt = 0
    kd = ab.shape[0] - 1
    while True:
        try:
            cb = sla.cholesky_banded(ab, lower=True, check_finite=False)
            if not np.all(np.isfinite(cb[0])) or np.any(cb[0] <= 0):
                raise np.linalg.LinAlgError('non-positive pivot')
            break
        except np.linalg.LinAlgError:
            if force_psd and attempt < attempts:
                ab[0] += eps
                attempt += 1
                eps *= 10
            else:
                raise
    n = ab.shape[1]
    ub = np.zeros_like(cb)
    for d in range(kd + 1):
        ub[kd - d, d:] = cb[d, :n - d]
    mean = sla.cho_solve_banded((cb, True), rhs, check_finite=False)
    x = mean + sla.solve_banded((0, kd), ub, z, check_finite=False)
    return x, mean, cb, attempt


def step_V(W, V, cw, sw, Delta, lam2, Tau2, z, order, force_psd=True, eps=1e-6,
           attempts=4, want_diag=False):
    """GaussianBTF._resample_V (factor.py:364-409) with explicit noise
    z [M, T, K] (t-major).  The exact per-column statistics are used (the
    reference's stale likelihood cache, SURVEY.md Q2, is NOT reproduced)."""
    M, T, K = V.shape
    A, b = col_stats(W, cw, sw)
    Vn = np.empty_like(V)
    diag = dict(mean=np.zeros((M, T, K)), retries=np.zeros(M, dtype=int), A=A, b=b)
    if want_diag:
        diag['band'] = []
        diag['chol'] = []
    for j in range(M):
        Pm = prior_band(Delta, lam2, Tau2[j])
        ab = assemble_band(A[j], Pm, order)
        x, mean, cb, nretry = mvn_from_band(ab, b[j].ravel(), z[j].ravel(), force_psd, eps, attempts)
        Vn[j] = x.reshape(T, K)
        diag['mean'][j] = mean.reshape(T, K)
        diag['retries'][j] = nretry
        if want_diag:
            diag['band'].append(ab)
            diag['chol'].append(cb)
    return Vn, diag


# ----------------------------------------------------------------------------
# likelihood-specific weights
# ----------------------------------------------------------------------------
def gaussian_weights(cnt, S, nu2):
    """c = cnt/nu2 and c*ybar = S/nu2 (factor.py:343-346, 355, 360)."""
    return cnt / nu2, S / nu2


def binomial_weights(Ysucc, Ntrials, omega):
    """Binomial pseudo-data (factor.py:437-445): weight omega, rhs y - n/2;
    cells with NaN y or NaN n are missing."""
    obs = ~(np.isnan(Ysucc) | np.isnan(Ntrials))
    kappa = np.where(obs, np.where(obs, Ysucc, 0.0) - np.where(obs, Ntrials, 0.0) / 2.0, 0.0)
    return np.where(obs, omega, 0.0), kappa


# ----------------------------------------------------------------------------
# negative-binomial dispersion   (factor.py:513-554)
# ----------------------------------------------------------------------------
def step_R(R, W, V, data, rdims, zs, us, rpropstdev=0.1, rstdev=1.0, want_margin=False):
    """NegativeBinomialBTF._resample_R with explicit noise: ``zs`` [nmh, *R.shape]
    standard normals, ``us`` [nmh, *R.shape] uniforms.  Returns (R, N), and with
    ``want_margin`` also min |u - prob| / prob over the chain's decisions (inf for none):
    how far the closest accept/reject decision was from a tie."""
    from scipy.special import gammaln
    data = np.asarray(data, dtype=float)
    if data.ndim == 3:
        data = data[..., None]
    R = np.array(R, dtype=float)[..., None].copy()
    logR = np.log(R)
    psi = np.einsum('nk,mtk->nmt', W, V).clip(-10, 10)
    P = (1.0 / (1.0 + np.exp(-psi)))[..., None]
    agg = [3] + sorted(rdims)[::-1]
    margin = np.inf
    for s in range(zs.shape[0]):
        cand_log = logR + rpropstdev * zs[s][..., None]
        cand = np.exp(cand_log)
        dprior = -(cand_log ** 2 - logR ** 2) / (2.0 * rstdev ** 2)
        ll = (gammaln(data + cand) - gammaln(cand) - gammaln(data + R) + gammaln(R)
              + (cand - R) * np.log(1 - P))
        for dim in agg:
            ll = np.nansum(ll, axis=dim)
        dprior = np.squeeze(dprior).reshape(ll.shape)
        prob = np.exp(np.clip(dprior + ll, -10, 1)).reshape(R.shape)
        u = us[s][..., None]
        acc = (u <= prob) & (cand > 1)
        margin = min(margin, float(np.min(np.abs(u - prob) / prob)))
        logR[acc] = cand_log[acc]
        R[acc] = np.exp(cand_log[acc])
    Ncount = np.nansum(data + R, axis=-1)
    if want_margin:
        return R[..., 0], Ncount, margin
    return R[..., 0], Ncount


# ----------------------------------------------------------------------------
# one full sweep (order: factor.py:306-311 then 112-128)
# ----------------------------------------------------------------------------
def gaussian_sweep(state, Y, noise, cfg):
    """One GaussianBTF.resample(Y).  ``state`` keys: W V Tau2 Tau2_a Tau2_b Tau2_c
    lam2 lam2_a sigma2 nu2.  ``noise`` keys: g_nu2, g_sigma2, g_tau [M,4,R_D],
    g_lam [2], z_W [N,K], z_V [M,T,K].  ``cfg`` keys: K, order, Delta, nu2_a/b,
    sigma2_a/b, stability, force_psd, force_psd_eps, force_psd_attempts,
    ref_compat, and optional sample_* flags.  Returns the new state dict."""
    st = dict(state)
    K, order, Delta = cfg['K'], cfg['order'], cfg['Delta']
    cnt, S, _ = prereduce(Y)
    if cfg.get('sample_nu2', True):
        st['nu2'] = step_nu2(st['W'], st['V'], Y, cfg['nu2_a'], cfg['nu2_b'], noise['g_nu2'])[0]
    if cfg.get('sample_sigma2', True):
        st['sigma2'] = step_sigma2(st['W'], cfg['sigma2_a'], cfg['sigma2_b'], noise['g_sigma2'])[0]
    if cfg.get('sample_Tau2', True):
        st['Tau2'], st['Tau2_a'], st['Tau2_b'], st['Tau2_c'] = step_tau2(
            st['V'], Delta, st['lam2'], st['Tau2_a'], st['Tau2_b'], st['Tau2_c'],
            noise['g_tau'], K, cfg['stability'])
    if cfg.get('sample_lam2', True):
        st['lam2'], st['lam2_a'] = step_lam2(st['V'], Delta, st['Tau2'], st['lam2_a'],
                                             noise['g_lam'], K, cfg.get('ref_compat', True))[:2]
    cw, sw = gaussian_weights(cnt, S, st['nu2'])
    if cfg.get('sample_W', True):
        st['W'] = step_W(st['W'], st['V'], cw, sw, st['sigma2'], noise['z_W'])[0]
    if cfg.get('sample_V', True):
        st['V'] = step_V(st['W'], st['V'], cw, sw, Delta, st['lam2'], st['Tau2'], noise['z_V'],
                         order, cfg['force_psd'], cfg['force_psd_eps'],
                         cfg['force_psd_attempts'])[0]
    return st


def binomial_sweep(state, Ysucc, Ntrials, noise, cfg):
    """One BinomialBTF.resample((Y, N)) (factor.py:437-460 + Gaussian W/V steps).
    ``noise['omega']`` is the [N,M,T] Polya-Gamma draw PG(N, W.V)."""
    st = dict(state)
    K, order, Delta = cfg['K'], cfg['order'], cfg['Delta']
    omega = noise['omega']
    with np.errstate(divide='ignore'):
        st['nu2'] = 1.0 / omega
    if cfg.get('sample_sigma2', True):
        st['sigma2'] = step_sigma2(st['W'], cfg['sigma2_a'], cfg['sigma2_b'], noise['g_sigma2'])[0]
    if cfg.get('sample_Tau2', True):
        st['Tau2'], st['Tau2_a'], st['Tau2_b'], st['Tau2_c'] = step_tau2(
            st['V'], Delta, st['lam2'], st['Tau2_a'], st['Tau2_b'], st['Tau2_c'],
            noise['g_tau'], K, cfg['stability'])
    if cfg.get('sample_lam2', True):
        st['lam2'], st['lam2_a'] = step_lam2(st['V'], Delta, st['Tau2'], st['lam2_a'],
                                             noise['g_lam'], K, cfg.get('ref_compat', True))[:2]
    cw, sw = binomial_weights(Ysucc, Ntrials, omega)
    if cfg.get('sample_W', True):
        st['W'] = step_W(st['W'], st['V'], cw, sw, st['sigma2'], noise['z_W'])[0]
    if cfg.get('sample_V', True):
        st['V'] = step_V(st['W'], st['V'], cw, sw, Delta, st['lam2'], st['Tau2'], noise['z_V'],
                         order, cfg['force_psd'], cfg['force_psd_eps'],
                         cfg['force_psd_attempts'])[0]
    return st
