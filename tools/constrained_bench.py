"""Sweeps/s of the constrained Poisson, Binomial or Gaussian model (ConstrainedNonconjugateBayesianTensorFiltering):
  politics   19 x 19 x 228, K = 5, p = 2, ngrid = 100 (the shape of politics/benchmark.py): the device path
             (loglikelihood='poisson', 'binomial' or 'gaussian', every step in the engine) and the host path (the same
             likelihood as a Python callable, GASS on the host), timed alternately in one process;
  large      1024 x 256 x 64, K = 8, device path only.
Poisson: synthetic counts from a positive low-rank rate, constraints Mu >= 0.  Binomial: 20 trials per cell, successes
from a low-rank probability in (0, 0.9], constraints 0 <= Mu <= 1.  Gaussian: the low-rank surface plus noise of sd
0.1, constraints Mu non-decreasing in t; the device samples nu2 every sweep, the host callable holds it at 0.01 (it
has no nu2 step).  Prints the card name and power limit beside the numbers.
usage: python tools/constrained_bench.py [--likelihood {poisson,binomial,gaussian}] [--rounds 2] [--steps 20]
       [--host-steps 20]"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests'))


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return q.stdout.strip()


def problem(N, M, T, K, seed, likelihood='poisson'):
    rs = np.random.RandomState(seed)
    W = np.abs(rs.normal(size=(N, K))) + 0.1
    W[np.triu_indices(K, k=1)] = 0
    V = (np.abs(rs.normal(size=(M, T, K))) * 0.2).cumsum(axis=1) / np.sqrt(T) + 0.05
    lam = np.einsum('nk,mtk->nmt', W, V)
    if likelihood == 'binomial':
        V *= 0.9 / lam.max()                   # p = W V^T in (0, 0.9]
        Nt = np.full(lam.shape, 20.0)
        Y = rs.binomial(20, np.einsum('nk,mtk->nmt', W, V)).astype(float)
        Y[rs.random_sample(Y.shape) < 0.1] = np.nan
        cons = np.concatenate([np.concatenate([np.eye(T), -np.eye(T)]),
                               np.concatenate([np.zeros(T), -np.ones(T)])[:, None]], axis=1)
        return W, V, (Y, Nt), cons
    if likelihood == 'gaussian':
        Y = lam + 0.1 * rs.normal(size=lam.shape)
        Y[rs.random_sample(Y.shape) < 0.1] = np.nan
        A = np.eye(T, k=1)[:-1] - np.eye(T)[:-1]      # Mu[t + 1] - Mu[t] >= 0
        return W, V, Y, np.concatenate([A, np.zeros((T - 1, 1))], axis=1)
    Y = rs.poisson(lam).astype(float)
    Y[rs.random_sample(Y.shape) < 0.1] = np.nan
    cons = np.concatenate([np.eye(T), np.zeros((T, 1))], axis=1)
    return W, V, Y, cons


def model(ll, N, M, T, K, W, V, cons, ngrid):
    from functionalmf_b200 import ConstrainedNonconjugateBayesianTensorFiltering as CM
    kw = dict(nu2_init=0.01) if ll == 'gaussian' else {}
    return CM(N, M, T, ll, cons, nembeds=K, tf_order=2, gass_ngrid=ngrid, W_init=W, V_init=V, seed=7, **kw)


def timed(m, Y, steps):
    m._engine.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        m.resample(Y)
    m._engine.synchronize()
    return (time.perf_counter() - t0) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--likelihood', choices=('poisson', 'binomial', 'gaussian'), default='poisson')
    ap.add_argument('--rounds', type=int, default=2)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--host-steps', type=int, default=20)
    args = ap.parse_args()
    warnings.simplefilter('ignore')
    lik = args.likelihood
    if lik == 'binomial':
        from test_gpu_constrained_binomial import binomial_rowcol_loglikelihood as host_ll
    elif lik == 'gaussian':
        from test_gpu_constrained_gaussian import GaussianLL
        host_ll = GaussianLL(0.01)
    else:
        from constrained_ll import rowcol_loglikelihood as host_ll
    out = {'card': card()}
    if lik != 'poisson':
        out['likelihood'] = lik
    N, M, T, K = 19, 19, 228, 5
    W, V, Y, cons = problem(N, M, T, K, 1, lik)
    dev = model(lik, N, M, T, K, W, V, cons, 100)
    host = model(host_ll, N, M, T, K, W, V, cons, 100)
    dev.run_gibbs(Y, nburn=3, nsamples=0, verbose=False)
    host.resample(Y)
    sec = {'device': [], 'host': []}
    for _ in range(args.rounds):
        # the device path as a chain (btf_run_segment / graph replay), the host path one resample per sweep
        dev._engine.synchronize()
        t0 = time.perf_counter()
        dev.run_gibbs(Y, nburn=args.steps, nsamples=0, verbose=False)
        sec['device'].append((time.perf_counter() - t0) / args.steps)
        sec['host'].append(timed(host, Y, args.host_steps))
    out['politics'] = {'shape': [N, M, T, K], 'ngrid': 100,
                       'device_sweeps_per_s': [round(1.0 / s, 2) for s in sec['device']],
                       'host_sweeps_per_s': [round(1.0 / s, 3) for s in sec['host']],
                       'device_resample_sweeps_per_s': round(1.0 / timed(dev, Y, args.steps), 2)}
    N, M, T, K = 1024, 256, 64, 8
    W, V, Y, cons = problem(N, M, T, K, 2, lik)
    big = model(lik, N, M, T, K, W, V, cons, 100)
    big.run_gibbs(Y, nburn=2, nsamples=0, verbose=False)
    s = []
    for _ in range(args.rounds):
        big._engine.synchronize()
        t0 = time.perf_counter()
        big.run_gibbs(Y, nburn=args.steps, nsamples=0, verbose=False)
        s.append((time.perf_counter() - t0) / args.steps)
    out['large'] = {'shape': [N, M, T, K], 'ngrid': 100, 'device_sweeps_per_s': [round(1.0 / x, 2) for x in s]}
    big._engine.enable_diag(True)
    big.resample(Y)
    out['large']['mean_feasible_W'] = float(big._engine.diag('gass_W')[:, 0].mean())
    out['large']['mean_feasible_V'] = float(big._engine.diag('gass_V')[:, 0].mean())
    print(json.dumps(out))


if __name__ == '__main__':
    main()
