"""Polya-Gamma sampler restated on the CPU (numpy).  TEST INFRASTRUCTURE ONLY.

The reference draws ``omega ~ PG(b, psi)`` through the third-party package
``pypolyagamma`` (factor.py:431-432, 459), which is NOT vendored in
/root/reference and is unpinned (setup.py:50): **parity unpinned**.  Upstream is
Linderman's wrapper of Windle's BayesLogit hybrid sampler.  This file restates
the published algorithms it is built from:

* PG(1, z): Devroye's exact alternating-series sampler, Polson, Scott & Windle
  (2013), "Bayesian inference for logistic models using Polya-Gamma latent
  variables", Algorithm 1 / BayesLogit ``rpg.devroye`` (truncation point
  t = 0.64, truncated inverse-Gaussian / exponential mixture proposal).
* PG(b, z), integer b: sum of b independent PG(1, z).
* PG(b, z), real b: floor(b) Devroye draws + the fractional part by the
  truncated sum-of-gammas series with its expected tail added back;
  b > 170: moment-matched normal approximation (the hybrid sampler's rule).

Validated by moments (tests/test_pg_oracle.py):
  E  = b/(2z) tanh(z/2),   Var = b/(4 z^3) (sinh z - z) sech^2(z/2)
                                = b/(4 z^3) (2 tanh(z/2) - z sech^2(z/2)).
"""
import numpy as np
from scipy.special import expit, log_ndtr

TRUNC = 0.64
PI = np.pi
NORMAL_B = 170.0          # b above which the normal approximation is used
SERIES_TERMS = 200        # truncated sum-of-gammas terms for the fractional part


def pg_mean(b, z):
    z = np.abs(np.asarray(z, dtype=float))
    small = z < 1e-6
    zs = np.where(small, 1.0, z)
    m = np.where(small, 0.25 * (1 - z * z / 12.0), np.tanh(zs / 2) / (2 * zs))
    return b * m


def pg_var(b, z):
    z = np.abs(np.asarray(z, dtype=float))
    small = z < 1e-3
    zs = np.where(small, 1.0, z)
    # (sinh z - z) sech^2(z/2) = 2 tanh(z/2) - z sech^2(z/2): no inf / inf past z = 710
    with np.errstate(over='ignore'):
        sech = 1.0 / np.cosh(zs / 2)
    v = (2 * np.tanh(zs / 2) - zs * sech * sech) / (4 * zs ** 3)
    v0 = (1.0 / 24.0) * (1 - z * z * (1.0 / 4.0 - 1.0 / 20.0))   # series around 0
    return b * np.where(small, v0, v)


def _a_coef(n, x):
    """Piecewise coefficient a_n(x) of the alternating series."""
    k = (n + 0.5) * PI
    with np.errstate(divide='ignore', over='ignore', invalid='ignore'):
        big = k * np.exp(-0.5 * k * k * x)
        sml = np.exp(-1.5 * (np.log(0.5 * PI) + np.log(x)) + np.log(k) - 2.0 * (n + 0.5) ** 2 / x)
    return np.where(x > TRUNC, big, sml)


def _mass_texpon(Z):
    fz = PI * PI / 8 + Z * Z / 2
    b = np.sqrt(1.0 / TRUNC) * (TRUNC * Z - 1)
    a = -np.sqrt(1.0 / TRUNC) * (TRUNC * Z + 1)
    x0 = np.log(fz) + fz * TRUNC
    xb = x0 - Z + log_ndtr(b)
    xa = x0 + Z + log_ndtr(a)
    # log(q/p) and p = 1 / (1 + q/p) = expit(-log(q/p)): q/p itself overflows for |z| > ~97, where p is 0
    log_qdivp = np.log(4 / PI) + np.logaddexp(xb, xa)
    return expit(-log_qdivp)


def _rtigauss(Z, rng):
    """Inverse-Gaussian(1/Z, 1) truncated to (0, TRUNC], vectorised rejection."""
    Z = np.asarray(Z, dtype=float)
    X = np.full(Z.shape, np.nan)
    todo = np.ones(Z.shape, dtype=bool)
    with np.errstate(divide='ignore'):
        mu = np.where(Z > 0, 1.0 / np.where(Z > 0, Z, 1.0), np.inf)
    while todo.any():
        idx = np.nonzero(todo)[0]
        z = Z[idx]
        m = mu[idx]
        x = np.empty(len(idx))
        ok = np.zeros(len(idx), dtype=bool)
        big = m > TRUNC
        # branch 1: mu > t -- exponential-tail proposal, accept with exp(-Z^2 X / 2)
        nb = int(big.sum())
        if nb:
            xb = np.empty(nb)
            need = np.ones(nb, dtype=bool)
            while need.any():
                k = int(need.sum())
                e1 = rng.exponential(size=k)
                e2 = rng.exponential(size=k)
                good = e1 * e1 <= 2 * e2 / TRUNC
                cand = TRUNC / (1 + TRUNC * e1) ** 2
                sel = np.nonzero(need)[0]
                xb[sel[good]] = cand[good]
                need[sel[good]] = False
            alpha = np.exp(-0.5 * z[big] ** 2 * xb)
            acc = rng.random(nb) <= alpha
            x[big] = xb
            ok[big] = acc
        # branch 2: mu <= t -- plain inverse-Gaussian draws until below t
        ns = int((~big).sum())
        if ns:
            ms = m[~big]
            y = rng.standard_normal(ns) ** 2
            xs = ms + 0.5 * ms * ms * y - 0.5 * ms * np.sqrt(4 * ms * y + (ms * y) ** 2)
            flip = rng.random(ns) > ms / (ms + xs)
            xs = np.where(flip, ms * ms / xs, xs)
            x[~big] = xs
            ok[~big] = xs <= TRUNC
        X[idx[ok]] = x[ok]
        todo[idx[ok]] = False
    return X


def pg1(z, rng):
    """Exact PG(1, z) draws for an array of tilts z (Devroye)."""
    z = np.asarray(z, dtype=float).ravel()
    Z = np.abs(z) * 0.5
    fz = PI * PI / 8 + Z * Z / 2
    out = np.empty(len(z))
    todo = np.ones(len(z), dtype=bool)
    pmass = _mass_texpon(Z)
    while todo.any():
        idx = np.nonzero(todo)[0]
        Zi = Z[idx]
        use_exp = rng.random(len(idx)) < pmass[idx]
        X = np.empty(len(idx))
        ne = int(use_exp.sum())
        if ne:
            X[use_exp] = TRUNC + rng.exponential(size=ne) / fz[idx][use_exp]
        if ne < len(idx):
            X[~use_exp] = _rtigauss(Zi[~use_exp], rng)
        S = _a_coef(0, X)
        Y = rng.random(len(idx)) * S
        n = 0
        undecided = np.ones(len(idx), dtype=bool)
        accepted = np.zeros(len(idx), dtype=bool)
        while undecided.any():
            n += 1
            an = _a_coef(n, X)
            if n % 2 == 1:
                S = np.where(undecided, S - an, S)
                acc = undecided & (Y <= S)
                accepted |= acc
                undecided &= ~acc
            else:
                S = np.where(undecided, S + an, S)
                rej = undecided & (Y > S)
                undecided &= ~rej
            if n > 200:            # numerically never reached
                break
        out[idx[accepted]] = 0.25 * X[accepted]
        todo[idx[accepted]] = False
    return out


def pg_frac(bf, z, rng):
    """PG(bf, z) for 0 < bf < 1: truncated sum of gammas + expected tail."""
    bf = np.asarray(bf, dtype=float).ravel()
    z = np.asarray(z, dtype=float).ravel()
    k = np.arange(1, SERIES_TERMS + 1)[None, :] - 0.5
    d = 4 * PI * PI * k * k + (z * z)[:, None]
    g = rng.standard_gamma(np.broadcast_to(bf[:, None], d.shape))
    x = 2.0 * (g / d).sum(axis=1)
    # expected remainder: E[PG(bf,z)] minus the mean of the K retained terms
    # (sum_{k>=1} 1/(4 pi^2 (k-1/2)^2 + z^2) = tanh(z/2)/(4z) in closed form)
    tail = pg_mean(bf, z) - 2.0 * bf * (1.0 / d).sum(axis=1)
    return x + tail


def pgdraw(b, z, rng):
    """PG(b, z) for arrays b >= 0 (real) and z; b <= 0 or non-finite -> 0."""
    b = np.asarray(b, dtype=float).ravel()
    z = np.asarray(z, dtype=float).ravel()
    out = np.zeros(len(b))
    valid = np.isfinite(b) & (b > 0) & np.isfinite(z)
    normal = valid & (b > NORMAL_B)
    if normal.any():
        m = pg_mean(b[normal], z[normal])
        v = pg_var(b[normal], z[normal])
        out[normal] = m + np.sqrt(v) * rng.standard_normal(int(normal.sum()))
    rest = valid & ~normal
    if rest.any():
        idx = np.nonzero(rest)[0]
        bi = np.floor(b[idx]).astype(np.int64)
        bf = b[idx] - bi
        acc = np.zeros(len(idx))
        # integer part: repeat PG(1) draws for the cells that still need one
        rep = np.repeat(np.arange(len(idx)), bi)
        if len(rep):
            draws = pg1(z[idx][rep], rng)
            np.add.at(acc, rep, draws)
        fr = bf > 1e-12
        if fr.any():
            acc[fr] += pg_frac(bf[fr], z[idx][fr], rng)
        out[idx] = acc
    return out
