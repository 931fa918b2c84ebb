"""ConstrainedNonconjugateBayesianTensorFiltering (factor.py:894-1017) on the B200 engine.

The likelihood is an arbitrary Python callable and the W / V updates are generalized analytic
slice sampling under linear constraints (factor.py:665-892, gass.py:13-130), so the slice
sampling itself stays on the host -- exactly one Python likelihood call per row / column and
candidate batch, as in the reference.  Everything that is linear algebra comes from the CUDA
engine in ONE batched launch per step instead of per-row / per-column Python + CHOLMOD calls:

* W step: for every row the EP-centred Gaussian  N(Q_i^-1 b_i, Q_i^-1)  (factor.py:678-687) --
  statistics kernel K1a with weights 1/Sigma_ep^2, batched Cholesky K2 -> conditional mean mu_i and
  the elliptical proposal v_i = L_i^-T z_i for all rows at once;
* V step: for every column the banded system  Q_j = Q_lik + kron(I, Delta^T diag(.) Delta)
  (factor.py:767-797, prior precision clipped to [stability, 1/stability]) -- K1b + K3 -> mu_j and
  v_j = L_j^-T z_j for all columns at once;
* sigma2 / Tau2 / lam2 steps (factor.py:130-153) run on the device as for the conjugate models.

``loglikelihood='poisson'`` selects the built-in Poisson likelihood of examples/poisson_tensor_filtering.py
(``nansum(poisson.logpmf(Y, W V^T))`` over the replicates).  ``loglikelihood='binomial'`` selects the built-in Binomial
likelihood of successes out of trials, ``data = (Y, Ntrials)``, whose success probability is the surface p = W V^T
itself (``nansum(binom.logpmf(Y, Ntrials, W V^T))``; the constraints keep p in [0, 1] and give it its shape).
``loglikelihood='gaussian'`` selects the Gaussian likelihood ``nansum(norm.logpdf(Y, W V^T, sqrt(nu2)))`` over the
replicates, for continuous responses with a shape-constrained mean; its noise variance ``nu2`` takes the arguments
and rules of GaussianBayesianTensorFiltering (``nu2_init``, ``nu2_true``, ``nu2_a``, ``nu2_b``): a scalar sampled from
its conjugate conditional at the start of every sweep, a fixed scalar, or fixed known per-cell variances [N, M, T].
It needs at least one constraint (on the tensor or on the rows of W): without any, W and V have Gaussian conditionals,
which GaussianBayesianTensorFiltering draws exactly, so the slice sampler would only mix more slowly; that
combination raises ValueError.  With any of the three built-in likelihoods, the whole sweep -- (nu2,) sigma2, Tau2, lam2, the W and V centres and proposals, and one GASS
transition per row and per column -- runs inside the engine (gass_kernels.cu), so
``run_gibbs`` runs in ``btf_run_segment`` pieces (or a CUDA graph) and ``HeldOutEvaluator``, ``track_mu``,
``results_dir`` and checkpoints work as for the conjugate models.  Its random choices are Philox draws of the engine,
not ``np.random``.  Single GPU.

``nthreads``, ``multiprocessing``, ``sharedprefix`` are accepted and ignored (there is no worker
pool to manage: rows and columns are batched on the GPU); ``shutdown()`` is a no-op kept for
drop-in compatibility.
"""
import warnings
import numpy as np
from scipy.stats import binom, norm, poisson

from . import _lib as L
from .factor import BayesianTensorFiltering, _BayesianModel, _GaussianNoise
from .gass import gass, FINE_GRID


class ConstrainedNonconjugateBayesianTensorFiltering(_GaussianNoise, BayesianTensorFiltering):
    # the engine runs in its f64-weight mode: weights = 1/Sigma_ep^2 are injected as "omega"
    _likelihood = L.BINOMIAL
    # the built-in likelihoods, whose GASS steps run on the device
    _BUILTIN = {'poisson': L.POISSON, 'binomial': L.CBINOMIAL, 'gaussian': L.CGAUSSIAN}

    def __init__(self, nrows, ncols, ndepth, loglikelihood, Constraints, ep_approx=None, nthreads=3,
                 gass_ngrid=100, Row_constraints=None, multiprocessing=True, sharedprefix=None,
                 worker_init=None, **kwargs):
        self._builtin = loglikelihood if isinstance(loglikelihood, str) else None
        if self._builtin is not None:
            if loglikelihood not in self._BUILTIN:
                raise ValueError("loglikelihood must be a callable, 'poisson', 'binomial' or 'gaussian', got %r"
                                 % (loglikelihood,))
            self._likelihood = self._BUILTIN[loglikelihood]
        self.loglikelihood = loglikelihood
        Constraints = np.asarray(Constraints, dtype=float)
        self.Constraints_A, self.Constraints_C = Constraints[:, :-1], Constraints[:, -1:]
        self.nconstraints = self.Constraints_A.shape[0]
        if self._builtin == 'gaussian' and self.nconstraints == 0 and (
                Row_constraints is None or np.size(Row_constraints) == 0):
            raise ValueError("loglikelihood='gaussian' without any constraint is the conjugate Gaussian model: use "
                             "GaussianBayesianTensorFiltering, which draws W and V from their exact conditionals")
        self.nthreads, self.gass_ngrid = nthreads, gass_ngrid
        self.Row_constraints = Row_constraints
        self.multiprocessing, self.sharedprefix = multiprocessing, sharedprefix
        if ep_approx is None:
            self.Mu_ep, self.Sigma_ep = None, None
        else:
            self.Mu_ep, self.Sigma_ep = ep_approx
        self._ep_key = None
        self._gass_key = None
        self._rng = np.random            # slice heights / grid choices: the reference's global stream
        super().__init__(nrows, ncols, ndepth, **kwargs)
        if worker_init is not None:
            worker_init(self)

    # ---- engine configuration
    def _gaussian_noise(self):
        return self._builtin == 'gaussian'      # nu2 (_GaussianNoise) exists for the built-in Gaussian likelihood only

    def _likelihood_options(self):
        opts = super()._likelihood_options()
        opts.update(clip_prior_precision=1)
        return opts

    def shutdown(self):
        """Nothing to release: the reference tears down its worker pool and shared memory here
        (factor.py:963-982)."""

    # ---- EP approximation -> engine pseudo-data: weights 1/Sigma^2, weighted sums Mu/Sigma^2
    def _sync_ep(self):
        N, M, T = self.nrows, self.ncols, self.ndepth
        key = None if self.Mu_ep is None else (self._fingerprint(self.Mu_ep), self._fingerprint(self.Sigma_ep))
        if self._builtin:
            if key != self._ep_key:
                self._ep_key = None
                if self.Mu_ep is None:
                    self._engine.set_ep(None, None)
                else:
                    self._engine.set_ep(np.asarray(self.Mu_ep, dtype=float), np.asarray(self.Sigma_ep, dtype=float))
                self._ep_key = key
            return
        if key == self._ep_key and self._omega is not None:
            return
        if self.Mu_ep is None:
            y = np.full((N, M, T), np.nan)
            self._omega = np.zeros((N, M, T))
        else:
            Mu, Sig = np.asarray(self.Mu_ep, dtype=float), np.asarray(self.Sigma_ep, dtype=float)
            obs = ~np.isnan(Mu)
            w = np.where(obs, 1.0 / np.where(obs, Sig, 1.0) ** 2, 0.0)
            y = np.where(obs, np.where(obs, Mu, 0.0) * w, np.nan)
            self._omega = w
        # engine pseudo-data: kappa = y - n/2 with n = 0
        self._engine.set_data_binomial(y, np.where(np.isnan(y), np.nan, 0.0))
        self._ep_key = key

    _omega = None

    def _sync_gass(self):
        """Constraints, row constraints and the angle grids of the device GASS steps (re-sent when they change)."""
        R = self.Row_constraints
        key = (int(self.gass_ngrid), self._fingerprint(self.Constraints_A), self._fingerprint(self.Constraints_C),
               None if R is None else self._fingerprint(R))
        if key == self._gass_key:
            return
        self._gass_key = None
        self._engine.set_gass(self.Constraints_A, self.Constraints_C[:, 0], np.linspace(-np.pi, np.pi, FINE_GRID),
                              np.linspace(-np.pi, np.pi, int(self.gass_ngrid)), rowcons=R)
        self._gass_key = key

    def _binomial_data(self, data):
        """(Y, Ntrials) of the built-in Binomial likelihood as two float arrays of the model's [N, M, T] shape."""
        shape = (self.nrows, self.ncols, self.ndepth)
        if isinstance(data, (tuple, list)) and len(data) == 2:
            Y, Nt = np.asarray(data[0], dtype=float), np.asarray(data[1], dtype=float)
            if Y.shape == shape and Nt.shape == shape:
                return Y, Nt
        raise ValueError("loglikelihood='binomial' takes the data as a tuple (Y, Ntrials) of two %r arrays" % (shape,))

    def _upload(self, data):
        if self._builtin == 'binomial':
            Y, Nt = self._binomial_data(data)
            full = getattr(self, '_full_check', False)
            key = (self._fingerprint(Y, full), self._fingerprint(Nt, full))
            self._data_nbytes = int(Y.nbytes + Nt.nbytes)
            if key != self._data_key:
                self._data_key = None
                self._engine.set_data_binomial(Y, Nt)
                self._data_key = key
            self._sync_gass()
        elif self._builtin in ('poisson', 'gaussian'):
            Y = np.asarray(data)
            assert Y.ndim in (3, 4), 'Observations must be a 3- or 4-tensor.'
            key = self._fingerprint(data, getattr(self, '_full_check', False))
            self._data_nbytes = int(Y.nbytes)
            if key != self._data_key:
                self._data_key = None
                if self._builtin == 'poisson':
                    self._engine.set_data_poisson(Y)
                else:
                    self._engine.set_data_gaussian(Y)
                self._data_key = key
            self._sync_gass()
        self._sync_ep()

    # ---- batched Gaussian centres / proposals from the engine
    def _engine_step(self, mask, z_name=None, z=None):
        eng = self._engine
        self._push_state()
        eng.set_sample_mask(mask)
        if mask & (L.SAMPLE_W | L.SAMPLE_V):
            eng.inject('omega', self._omega)
            if z is not None:
                eng.inject(z_name, z)
            eng.enable_diag(True)
        eng.sweep(1)

    def _device_hyper_step(self):
        mask = 0
        for flag, bit in (('sample_sigma2', L.SAMPLE_SIGMA2), ('sample_Tau2', L.SAMPLE_TAU2),
                          ('sample_lam2', L.SAMPLE_LAM2)):
            if getattr(self, flag, False):
                mask |= bit
        if mask:
            self._engine_step(mask)
            for name in ('Tau2', 'Tau2_a', 'Tau2_b', 'Tau2_c'):
                setattr(self, name, self._engine.get(name))
            for name in self._scalar_names():
                setattr(self, name, self._engine.get_scalar(name))

    def resample(self, data, **kwargs):
        '''One sweep: sigma2, Tau2, lam2 (device), then GASS for W and V (factor.py:112-128).'''
        if self._builtin:
            return BayesianTensorFiltering.resample(self, data, **kwargs)
        self._sync_ep()
        self._device_hyper_step()
        if self.sample_W:
            self._resample_W(data)
        if self.sample_V:
            self._resample_V(data)

    def run_gibbs(self, data, nburn=1000, nthin=1, nsamples=1000, verbose=True, print_freq=100,
                  callback=None, **kwargs):
        if self._builtin:
            return _BayesianModel.run_gibbs(self, data, nburn=nburn, nthin=nthin, nsamples=nsamples, verbose=verbose,
                                            print_freq=print_freq, callback=callback, **kwargs)
        # the likelihood is a Python callback: always the per-sweep path of genlasso.py:37-66
        cb = callback if callback is not None else (lambda *a, **k: None)
        return self._run_gibbs_callback(data, nburn, nthin, nsamples, verbose, print_freq, cb, **kwargs)

    # ---- W | rest  (factor.py:665-757)
    def _w_constraints(self, i):
        nd = min(self.nembeds, i + 1)
        A = (self.Constraints_A[None, :, :, None] * self.V[:, None])[..., :nd].sum(axis=2)   # [M, J, nd]
        C = np.tile(self.Constraints_C, (self.ncols, 1))
        cons = np.concatenate([A.reshape((-1, nd)), C], axis=1)
        if self.Row_constraints is not None:
            R = np.asarray(self.Row_constraints, dtype=float)
            cons = np.concatenate([cons, np.concatenate([R[:, :nd], R[:, -1:]], axis=1)], axis=0)
        return cons

    def _w_loglikelihood(self, w, ll_args):
        i, data, V_i, mu_ep, sigma_ep = ll_args
        if w.ndim > 1:
            tau = (V_i[None] * w[:, None, None]).sum(axis=-1)
            ll = np.array([self.loglikelihood(data, t, wk, V_i, row=i) for t, wk in zip(tau, w)])
            if mu_ep is not None:
                ll -= norm.logpdf(tau, mu_ep[None], sigma_ep[None]).sum(axis=-1).sum(axis=-1)
            return ll
        tau = (V_i * w[None, None]).sum(axis=-1)
        ll = self.loglikelihood(data, tau, w, V_i, row=i)
        if mu_ep is not None:
            ll -= norm.logpdf(tau, mu_ep, sigma_ep).sum()
        return ll

    def _resample_W(self, data, z=None):
        self._engine_step(L.SAMPLE_W, 'z_W', z)
        mean = self._engine.diag('W_mean')
        draw = self._engine.get('W')
        for i in range(self.nrows):
            nd = min(self.nembeds, i + 1)
            V_i = self.V[:, :, :nd]
            mu_ep = None if self.Mu_ep is None else self.Mu_ep[i]
            sg_ep = None if self.Mu_ep is None else self.Sigma_ep[i]
            mu_i = mean[i, :nd] if self.Mu_ep is not None else np.zeros(nd)
            self.W[i, :nd], _ = gass(self.W[i, :nd].copy(), draw[i, :nd] - mean[i, :nd], self._w_loglikelihood,
                                     self._w_constraints(i), mu=mu_i, ll_args=(i, data, V_i, mu_ep, sg_ep),
                                     ngrid=self.gass_ngrid, rng=self._rng)

    # ---- V | rest  (factor.py:759-892); vectors are k-major (x[k*T + t] = V[j,t,k]) as in the reference
    def _v_constraints(self):
        A = (self.Constraints_A[None, :, None, :] * self.W[:, None, :, None]).reshape(
            (self.nrows * self.nconstraints, self.nembeds * self.ndepth))
        C = np.tile(self.Constraints_C, (self.nrows, 1))
        return np.concatenate([A, C], axis=1)

    def _v_loglikelihood(self, v, ll_args):
        j, data, mu_ep, sigma_ep = ll_args
        if v.ndim > 1:
            Vb = np.transpose(v.reshape((-1, self.nembeds, self.ndepth)), [0, 2, 1])
            tau = (Vb[:, None] * self.W[None, :, None]).sum(axis=-1)
            ll = np.array([self.loglikelihood(data, t, self.W, vk, col=j) for t, vk in zip(tau, Vb)])
            if mu_ep is not None:
                ll -= norm.logpdf(tau, mu_ep[None], sigma_ep[None]).sum(axis=-1).sum(axis=-1)
            return ll
        Vj = v.reshape((self.nembeds, self.ndepth)).T
        tau = (Vj[None] * self.W[:, None]).sum(axis=-1)
        ll = self.loglikelihood(data, tau, self.W, Vj, col=j)
        if mu_ep is not None:
            ll -= norm.logpdf(tau, mu_ep, sigma_ep).sum()
        return ll

    def _resample_V(self, data, z=None):
        self._engine_step(L.SAMPLE_V, 'z_V', z)
        mean = self._engine.diag('V_mean')
        draw = self._engine.get('V')
        cons = self._v_constraints()
        for j in range(self.ncols):
            mu_ep = None if self.Mu_ep is None else self.Mu_ep[:, j]
            sg_ep = None if self.Mu_ep is None else self.Sigma_ep[:, j]
            x = self.V[j].T.flatten()
            mu_j = mean[j].T.flatten() if self.Mu_ep is not None else np.zeros_like(x)
            v_j = (draw[j] - mean[j]).T.flatten()
            xn, _ = gass(x, v_j, self._v_loglikelihood, cons, mu=mu_j, ll_args=(j, data, mu_ep, sg_ep),
                         ngrid=self.gass_ngrid, rng=self._rng)
            self.V[j] = xn.reshape((self.nembeds, self.ndepth)).T

    def _finish_results(self, results):
        results = super()._finish_results(results)
        results.pop('_nu2_scalar', None)         # (the built-in Gaussian likelihood has made it results['nu2'])
        return results

    def logprob(self, data, **kwargs):
        tau = (self.W[:, None, None] * self.V[None]).sum(axis=-1)
        if self._builtin:
            with warnings.catch_warnings():
                warnings.simplefilter('ignore', category=RuntimeWarning)
                if self._builtin == 'binomial':
                    Y, Nt = self._binomial_data(data)
                    return np.nansum(binom.logpmf(Y, Nt, tau))
                Y = np.asarray(data)
                if Y.ndim > tau.ndim:
                    tau = tau[..., None]
                if self._builtin == 'gaussian':
                    nu2 = np.asarray(self.nu2, dtype=float)
                    if nu2.ndim and Y.ndim > nu2.ndim:
                        nu2 = nu2[..., None]
                    Y = np.where(np.isinf(nu2), np.nan, Y)          # a known variance of +inf: the cell is missing
                    return np.nansum(norm.logpdf(Y, tau, np.sqrt(nu2)))
                return np.nansum(poisson.logpmf(Y, tau))
        return self.loglikelihood(data, tau, self.W, self.V)


class NonconjugateBayesianTensorFiltering(ConstrainedNonconjugateBayesianTensorFiltering):
    """factor.py:567-612: black-box likelihood ``loglikelihood(W, V, data)``, joint elliptical slice
    sampling of all free W entries, then of all of V.  The prior draws the ellipse needs --
    W ~ N(0, sigma2) on the free entries (factor.py:155-174) and one banded MVN draw per column
    (factor.py:176-194, unclipped prior precision) -- come from the engine in one batched step each;
    the slice sampling itself and the likelihood callback stay on the host as in the reference."""

    def __init__(self, nrows, ncols, ndepth, loglikelihood, **kwargs):
        if isinstance(loglikelihood, str):
            raise ValueError('NonconjugateBayesianTensorFiltering takes a callable loglikelihood(W, V, data)')
        no_constraints = np.zeros((0, ndepth + 1))
        super().__init__(nrows, ncols, ndepth, loglikelihood, no_constraints, **kwargs)

    def _likelihood_options(self):
        return dict(clip_prior_precision=0)

    def _free_mask(self):
        m = np.ones((self.nrows, self.nembeds), dtype=bool)
        d = min(self.nrows, self.nembeds)
        iu = np.triu_indices(d, k=1, m=self.nembeds)
        m[:d][iu] = False
        return m

    def _resample_W(self, data, z=None):
        from .ess import elliptical_slice
        self._engine_step(L.SAMPLE_W, 'z_W', z)
        prior = self._engine.get('W')
        free = self._free_mask()

        def ll(vec, args):
            W = np.zeros_like(self.W)
            W[free] = vec
            return self.loglikelihood(W, self.V, args)
        new, _ = elliptical_slice(self.W[free], prior[free], ll, ll_args=data, rng=self._rng)
        self.W[free] = new

    def _resample_V(self, data, z=None):
        from .ess import elliptical_slice
        self._engine_step(L.SAMPLE_V, 'z_V', z)
        prior = self._engine.get('V')

        def ll(vec, args):
            return self.loglikelihood(self.W, vec.reshape(self.V.shape), args)
        new, _ = elliptical_slice(self.V.ravel(), prior.ravel(), ll, ll_args=data, rng=self._rng)
        self.V[:] = new.reshape(self.V.shape)

    def logprob(self, data, **kwargs):
        return self.loglikelihood(self.W, self.V, data)
