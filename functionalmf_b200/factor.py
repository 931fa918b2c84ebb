"""Drop-in sampler classes of functionalmf/factor.py backed by the B200 engine.

Same constructors, attributes (``W, V, Tau2, lam2, sigma2, nu2, R, Delta`` ...),
``resample(data)``, ``inferred_variables()`` and ``run_gibbs(...)`` result dict as
the reference (factor.py:23-563, genlasso.py:31-66); every numerical step of the
sweep runs in hand-written sm_100a CUDA through the C ABI of ``include/btf_b200.h``.
There is no CPU path: constructing a model without the CUDA library / a GPU raises.

Differences, all deliberate (SURVEY.md appendix D):
* randomness is Philox on the device, seeded from ``np.random`` at construction
  (so ``np.random.seed(s)`` still makes a run reproducible) or from ``seed=``;
* the V step uses the exact per-column statistics (no stale likelihood cache, Q2/Q3);
* Cholesky retries are bounded and raise ``NotPositiveDefiniteError`` (Q4/Q5);
* ``Tau2_init`` / ``Tau2_true`` still initialise ``Tau2_a/b/c`` from the prior (Q6);
* ``lam2`` follows the reference as written (last column only, Q1) unless
  ``ref_compat=False``;
* with known per-cell noise variances (Gaussian ``nu2`` an [N, M, T] array held
  fixed, also for the constrained model's ``'gaussian'`` likelihood), ``run_gibbs`` returns ``results['nu2']`` as a read-only
  ``np.broadcast_to`` view [nsamples, N, M, T] of that one array, not nsamples
  copies.
"""
import warnings
import numpy as np

from . import _lib as L
from .engine import Engine, pinned_empty
from .utils import ilogit  # noqa: F401  (re-exported like the reference module)

_ENGINE_KW = ('seed', 'device', 'ref_compat', 'shard', 'use_graph', 'resid_direct',
              'stats_splits_row', 'stats_splits_col', 'pinned_results')


class _BayesianModel(object):
    """run_gibbs / inferred_variables of functionalmf/genlasso.py:5-66."""

    def __init__(self, **kwargs):
        pass   # unknown keyword arguments (e.g. nthreads) are swallowed like the reference

    def inferred_variables(self):
        '''All non-nuisance parameters inferred by calling resample.'''
        results = {}
        self._inferred_variables(results)
        return results

    def run_gibbs(self, data, nburn=1000, nthin=1, nsamples=1000, verbose=True, print_freq=100,
                  callback=None, track_mu=False, results_dir=None, **kwargs):
        '''Run a gibbs sampler on the model (genlasso.py:37-66).  ``track_mu=True`` (engine
        extension) additionally returns ``results['Mu_mean']`` / ``results['Mu_var']``: the
        posterior mean and variance of einsum('nk,mtk->nmt', W, V) over the saved samples,
        accumulated on the device.  ``results_dir=path`` (engine extension) keeps the saved samples of W, V and
        Tau2 in ``path/<name>.npy`` (memory-mapped, written as the chain runs) instead of host memory:
        a thousand samples of the 4096 x 1024 x 64 configuration are 10 GB (SURVEY.md 8f row 2).'''
        nsteps = nburn + nthin * nsamples
        if callback is not None:
            return self._run_gibbs_callback(data, nburn, nthin, nsamples, verbose, print_freq, callback, **kwargs)
        self._full_check = True          # one whole-buffer checksum per chain
        try:
            self._begin(data)
        finally:
            self._full_check = False
        if track_mu:
            self._engine.track_mu_stats(True)
        for ev in getattr(self, '_evaluators', {}).values():
            ev._arm(nsamples)        # HeldOutEvaluator (metrics.py): every saved sample is scored on the device
        self._results_dir = results_dir
        results = self._alloc_results(nsamples)
        self._results_dir = None
        outs = self._result_buffers(results)
        seg = max(1, int(print_freq)) if verbose else nsteps
        step = 0
        while step < nsteps:
            if verbose and step % print_freq == 0:
                print('\tStep {}'.format(step))
            stop = min(nsteps, (step // seg + 1) * seg)
            # first saved step at or after `step`
            first = max(step, nburn)
            first = nburn + -(-(first - nburn) // nthin) * nthin
            if first < stop and nsamples > 0:
                self._engine.run_segment(stop - step, first - step, nthin, (first - nburn) // nthin, **outs)
            else:
                self._engine.sweep(stop - step)
            step = stop
        self._end()
        results = self._finish_results(results)
        for val in results.values():
            if isinstance(val, np.memmap):
                val.flush()
        if track_mu:
            results['Mu_mean'], results['Mu_var'], _ = self._engine.mu_stats()
            self._engine.track_mu_stats(False)
        return results

    def _run_gibbs_callback(self, data, nburn, nthin, nsamples, verbose, print_freq, callback, **kwargs):
        nsteps = nburn + nthin * nsamples
        results = None
        evaluators = list(getattr(self, '_evaluators', {}).values())
        for ev in evaluators:
            ev._arm(nsamples)
        for step in range(nsteps):
            if verbose and step % print_freq == 0:
                print('\tStep {}'.format(step))
            self.resample(data, **kwargs)
            callback(self, data, step, **kwargs)
            if getattr(self, '_data_nbytes', 0) > self.full_checksum_bytes:
                self.invalidate_data()       # a callback may edit a large array in place: never trust the sample
            if step >= nburn and (step - nburn) % nthin == 0:
                sidx = (step - nburn) // nthin
                inferred = self.inferred_variables()
                if results is None:
                    results = {}
                    for key, val in inferred.items():
                        results[key] = np.zeros([nsamples] + ([1] if np.isscalar(val) else list(np.shape(val))))
                for key, val in inferred.items():
                    results[key][sidx] = val
                for ev in evaluators:
                    ev.update()
        return results


class BayesianTensorFiltering(_BayesianModel):
    _likelihood = None

    def __init__(self, nrows, ncols, ndepth,
                 nembeds=5, tf_order=2,
                 sigma2_init=None, sigma2_true=None,
                 sigma2_a=0.1, sigma2_b=0.1,
                 lam2_init=None, lam2_true=None,
                 Tau2_init=None, Tau2_true=None,
                 W_init=None, V_init=None,
                 W_true=None, V_true=None,
                 stability=1e-6,
                 force_psd=True,
                 force_psd_eps=1e-6,
                 force_psd_attempts=4,
                 **kwargs):
        eng_kw = {k: kwargs.pop(k) for k in list(kwargs) if k in _ENGINE_KW}
        super().__init__(**kwargs)
        if self._likelihood is None:
            raise NotImplementedError('use one of the likelihood-specific subclasses')
        self.nrows, self.ncols, self.ndepth, self.nembeds = nrows, ncols, ndepth, nembeds
        self.tf_order = tf_order
        self.stability = stability
        self.linalg_opts = dict(force_psd=force_psd, force_psd_eps=force_psd_eps,
                                force_psd_attempts=force_psd_attempts)
        self.sigma2_a, self.sigma2_b = sigma2_a, sigma2_b
        self._pinned_results = bool(eng_kw.pop('pinned_results', True))
        self._shard = eng_kw.pop('shard', None)
        seed = eng_kw.pop('seed', None)
        if seed is None:
            seed = int(np.random.randint(0, 2 ** 31 - 1)) * 2654435761 % (2 ** 63)
        sharded = self._shard is not None and self._shard.world_size > 1
        if sharded:
            # sigma2, nu2, lam2 and the Tau2 chain are replicated, not communicated: every rank must run the same
            # Philox key.  Rank 0's seed wins (a per-process np.random draw would differ from rank to rank).
            from .distributed import agree_seed
            seed = agree_seed(int(seed))
        opts = dict(sigma2_a=sigma2_a, sigma2_b=sigma2_b, stability=stability,
                    force_psd=int(bool(force_psd)), force_psd_eps=force_psd_eps,
                    force_psd_attempts=int(force_psd_attempts), seed=int(seed),
                    ref_compat_lam2=int(bool(eng_kw.pop('ref_compat', True))))
        opts.update(self._likelihood_options())
        if self._shard is not None:
            opts.update(self._shard.engine_options())
        for k in ('device', 'use_graph', 'resid_direct', 'stats_splits_row', 'stats_splits_col'):
            if k in eng_kw:
                opts[k] = int(eng_kw[k])
        self._engine = Engine(nrows, ncols, ndepth, nembeds=nembeds, tf_order=tf_order,
                              likelihood=self._likelihood, **opts)
        if self._shard is not None and self._shard.world_size > 1:
            from .distributed import agree_unique_id
            self._engine.nccl_init(agree_unique_id())
        self._data_key = None
        eng = self._engine

        # Setup the trend filtering prior (factor.py:50)
        from scipy.sparse import csc_matrix
        self.Delta = csc_matrix(eng.get('Delta'))

        # ---- initial state, same precedence as factor.py:52-110
        init = 0
        self.sample_sigma2 = sigma2_true is None
        if sigma2_true is not None:
            eng.set('sigma2', [sigma2_true])
        elif sigma2_init is not None:
            eng.set('sigma2', [sigma2_init])
        else:
            init |= L.INIT_SIGMA2
        self.sample_lam2 = lam2_true is None
        init |= L.INIT_LAM2                       # _init_lam2 is always called for lam2_a (factor.py:72)
        self.sample_Tau2 = Tau2_true is None
        init |= L.INIT_TAU2                       # Tau2_a/b/c always exist (reference bug Q6)
        self.sample_W = W_true is None
        if W_true is None and W_init is None:
            init |= L.INIT_W
        self.sample_V = V_true is None
        init |= self._extra_init_mask()
        eng.init_state(init & ~L.INIT_V)
        if lam2_true is not None:
            eng.set('lam2', [lam2_true])
        elif lam2_init is not None:
            eng.set('lam2', [lam2_init])
        fixed_tau = Tau2_true if Tau2_true is not None else Tau2_init
        if fixed_tau is not None:
            fixed_tau = np.asarray(fixed_tau, dtype=float)
            assert fixed_tau.shape == (ncols, self.Delta.shape[0])
            eng.set('Tau2', fixed_tau)
        fixed_W = W_true if W_true is not None else W_init
        if fixed_W is not None:
            fixed_W = np.asarray(fixed_W, dtype=float)
            assert fixed_W.shape == (nrows, nembeds)
            eng.set('W', fixed_W)
        fixed_V = V_true if V_true is not None else V_init
        if fixed_V is not None:
            fixed_V = np.asarray(fixed_V, dtype=float)
            assert fixed_V.shape == (ncols, ndepth, nembeds)
            eng.set('V', fixed_V)
        else:
            eng.init_state(L.INIT_V)              # prior MVN draw per column (factor.py:235-242)
        self._after_base_init()
        self._pull_state()
        if sharded:
            # user-supplied *_init / *_true arrays must agree too: the sweep exchanges only the owned blocks
            from .distributed import assert_same_on_all_ranks
            assert_same_on_all_ranks(
                [self.W, self.V, self.Tau2, self.Tau2_a, self.Tau2_b, self.Tau2_c] +
                [np.asarray([float(np.ravel(getattr(self, n))[0]) for n in self._scalar_names()])],
                what='initial state (W, V, Tau2 chain, scalars)')

    # ---- hooks for subclasses
    def _likelihood_options(self):
        return {}

    def _extra_init_mask(self):
        return 0

    def _after_base_init(self):
        pass

    def _scalar_names(self):
        return ['sigma2', 'lam2', 'lam2_a']

    def _nu2_per_cell(self):
        """The known per-cell noise variances [N, M, T] the next sweep uses, or None (GaussianBayesianTensorFiltering)."""
        return None

    # ---- host <-> device coherence: the host attributes are authoritative between
    # calls (callers assign model.W[:] = ...), the device during a call
    def _push_state(self):
        eng = self._engine
        for name in ('W', 'V', 'Tau2', 'Tau2_a', 'Tau2_b', 'Tau2_c'):
            eng.set(name, getattr(self, name))
        for name in self._scalar_names():
            eng.set(name, [float(np.ravel(getattr(self, name))[0])])
        eng.set_sample_mask(self._sample_mask())

    def _pull_state(self):
        eng = self._engine
        for name in ('W', 'V', 'Tau2', 'Tau2_a', 'Tau2_b', 'Tau2_c'):
            setattr(self, name, eng.get(name))
        for name in self._scalar_names():
            setattr(self, name, eng.get_scalar(name))

    def _sample_mask(self):
        m = 0
        for flag, bit in (('sample_sigma2', L.SAMPLE_SIGMA2), ('sample_Tau2', L.SAMPLE_TAU2),
                          ('sample_lam2', L.SAMPLE_LAM2), ('sample_W', L.SAMPLE_W), ('sample_V', L.SAMPLE_V),
                          ('sample_nu2', L.SAMPLE_NU2), ('sample_R', L.SAMPLE_R)):
            if getattr(self, flag, False):
                m |= bit
        return m

    def _local_rows(self, arr):
        """Slice a full tensor down to this rank's row block (sharded engines)."""
        if self._shard is None or arr.shape[0] == self._engine.nloc != self.nrows:
            return arr
        if arr.shape[0] == self.nrows:
            r0, r1 = self._shard.rows
            return arr[r0:r1]
        return arr

    # ---- device copy of the data: re-uploaded whenever the array the caller passes has changed.
    # The reference reads ``data`` afresh on every call (factor.py:306-311); the engine keeps the compact
    # pre-reduction of it in HBM, so "has it changed" is decided by a checksum over the WHOLE buffer
    # (sum and xor of the 64-bit patterns: any single-element edit changes it), not by sampling:
    #   * run_gibbs: always the full checksum, once per chain;
    #   * resample(): the full checksum for arrays up to ``full_checksum_bytes`` (256 MB, ~30 ms); above that one
    #     checksum pass per sweep would cost more than the sweep itself, so a 2^20-element strided sample is used
    #     and in-place edits of larger arrays must be announced with ``model.invalidate_data()``.
    full_checksum_bytes = 256 << 20

    def invalidate_data(self):
        """Forget the device copy of the data: the next resample / run_gibbs uploads it again."""
        self._data_key = None

    @classmethod
    def _fingerprint(cls, arr, full=False):
        a = np.asarray(arr)
        if a.dtype != np.float64 or not a.flags.c_contiguous:
            a = np.ascontiguousarray(a, dtype=np.float64)
        bits = a.reshape(-1).view(np.uint64)
        if not full and a.nbytes > cls.full_checksum_bytes:
            bits = bits[::max(1, bits.size >> 20)]
        with np.errstate(over='ignore'):
            return (a.shape, int(bits.size), int(np.add.reduce(bits, dtype=np.uint64)),
                    int(np.bitwise_xor.reduce(bits)) if bits.size else 0)

    def _begin(self, data):
        self._upload(data)
        self._push_state()

    def _end(self):
        self._pull_state()

    def resample(self, data, **kwargs):
        '''One Gibbs sweep (factor.py:112-128 and the subclass overrides).'''
        self._begin(data)
        self._engine.sweep(1)
        self._end()

    # ---- checkpoint / resume (SURVEY.md section 5: the reference has none; a 12 h chain on 8 GPUs wants one)
    _CKPT_ARRAYS = ('W', 'V', 'Tau2', 'Tau2_a', 'Tau2_b', 'Tau2_c')

    def save_checkpoint(self, path):
        """Everything a chain needs to continue bit for bit: the state arrays and scalars, the Philox seed and the sweep
        counter (a Philox counter word), plus R for the negative-binomial model.  One ``.npz`` file; on a sharded model
        every rank holds the same state, so rank 0's file is enough."""
        eng = self._engine
        out = {k: eng.get(k) for k in self._CKPT_ARRAYS}
        for k in self._scalar_names():
            out[k] = np.array(eng.get_scalar(k))
        out['sweep'] = np.array(eng.get_scalar('sweep'))
        out['resid'] = np.array(eng.get_scalar('resid'))      # Gaussian: residual sum of the saved (W, V), input of the next nu2 step
        out['seed'] = np.array(int(eng.cfg.seed), dtype=np.uint64)
        if getattr(eng.cfg, 'likelihood', 0) == L.NEGBINOMIAL:
            out['R'] = eng.get('R')
        np.savez(path, **out)

    def load_checkpoint(self, path):
        """Restore a state written by ``save_checkpoint`` into a model built with the same shape and ``seed``; the next
        sweep is the one the saved chain would have run."""
        z = np.load(path)
        eng = self._engine
        if int(z['seed']) != int(eng.cfg.seed):
            raise ValueError('checkpoint was written with seed %d, this model has seed %d: pass seed=%d to the constructor'
                             % (int(z['seed']), int(eng.cfg.seed), int(z['seed'])))
        for k in self._CKPT_ARRAYS:
            if z[k].shape != eng.state_shape(k):
                raise ValueError('checkpoint %s has shape %r, the model expects %r' % (k, z[k].shape, eng.state_shape(k)))
            eng.set(k, z[k])
        for k in self._scalar_names():
            eng.set(k, [float(z[k])])
        if 'R' in z.files:
            eng.set('R', z['R'])
        eng.set('sweep', [float(z['sweep'])])
        if self._data_key is not None and 'resid' in z.files:
            eng.set('resid', [float(z['resid'])])              # after W and V (which invalidate it); needs the data on the device
        self._pull_state()
        if 'R' in z.files and hasattr(self, 'R'):
            self.R = eng.get('R')

    # ---- results
    def _alloc_results(self, nsamples):
        host = pinned_empty if self._pinned_results else (lambda s: np.empty(s, dtype=np.float64))
        spill = getattr(self, '_results_dir', None)

        def alloc(name, shape):
            if spill is None:
                return host(shape)
            import os
            os.makedirs(spill, exist_ok=True)
            return np.lib.format.open_memmap(os.path.join(spill, name + '.npy'), mode='w+', dtype=np.float64,
                                             shape=tuple(shape))
        res = {
            'W': alloc('W', (nsamples, self.nrows, self.nembeds)),
            'V': alloc('V', (nsamples, self.ncols, self.ndepth, self.nembeds)),
            'Tau2': alloc('Tau2', (nsamples, self.ncols, self.Delta.shape[0])),
            '_scalars': host((nsamples, 4)),
        }
        return res

    def _result_buffers(self, results):
        return dict(W=results['W'], V=results['V'], Tau2=results['Tau2'], scalars=results['_scalars'])

    def _finish_results(self, results):
        sc = results.pop('_scalars')
        results['sigma2'] = sc[:, 0:1].copy()
        results['lam2'] = sc[:, 1:2].copy()
        results['_nu2_scalar'] = sc[:, 2:3].copy()
        return results

    def _inferred_variables(self, var_map):
        var_map['W'] = np.copy(self.W)
        var_map['V'] = np.copy(self.V)
        var_map['sigma2'] = self.sigma2
        var_map['lam2'] = self.lam2
        var_map['Tau2'] = np.copy(self.Tau2)

    # the reference scripts call these to re-draw from the prior
    def _init_sigma2(self):
        self._engine.init_state(L.INIT_SIGMA2)
        self.sigma2 = self._engine.get_scalar('sigma2')

    def _init_lam2(self):
        self._engine.init_state(L.INIT_LAM2)
        self.lam2, self.lam2_a = self._engine.get_scalar('lam2'), self._engine.get_scalar('lam2_a')

    def _init_Tau2(self):
        self._engine.init_state(L.INIT_TAU2)
        for name in ('Tau2', 'Tau2_a', 'Tau2_b', 'Tau2_c'):
            setattr(self, name, self._engine.get(name))

    def _init_W(self):
        self._engine.set('sigma2', [float(self.sigma2)])
        self._engine.init_state(L.INIT_W)
        self.W = self._engine.get('W')

    def _init_V(self):
        self._engine.set('lam2', [float(self.lam2)])
        self._engine.set('Tau2', self.Tau2)
        self._engine.init_state(L.INIT_V)
        self.V = self._engine.get('V')

    @property
    def kernel_launches(self):
        return self._engine.kernel_launches


class _GaussianNoise(object):
    """The noise variance ``nu2`` of a Gaussian likelihood (factor.py:286-423), shared by
    GaussianBayesianTensorFiltering and the constrained model's built-in ``'gaussian'`` likelihood.

    ``nu2`` is a scalar, or an [N, M, T] array of known per-cell noise variances (the reference's heteroskedastic
    branch, e.g. per-cell standard errors squared): when ``model.nu2`` has that shape and ``sample_nu2`` is False
    (``nu2_true=array``), every cell is weighted by its own variance.  A variance of +inf makes an observed cell count
    as missing; NaN or <= 0 at an observed cell is refused.  With ``sample_nu2`` True the nu2 step draws a scalar from
    the residual like the reference's ``_resample_nu2``.  Single GPU only.

    A class that mixes this in and has other likelihoods too answers ``_gaussian_noise()`` with False for them: every
    hook below then defers to the next class in the MRO."""

    def __init__(self, nrows, ncols, ndepth, nu2_init=None, nu2_true=None, nu2_a=0.1, nu2_b=0.1, **kwargs):
        self.nu2_a, self.nu2_b = nu2_a, nu2_b
        self._nu2_args = (nu2_init, nu2_true)
        self._nu2_key = None          # fingerprint of the per-cell variances on the device, None in scalar mode
        super().__init__(nrows, ncols, ndepth, **kwargs)
        fixed = nu2_true if nu2_true is not None else nu2_init
        if self._nu2_cells_model() and fixed is not None and np.size(fixed) != 1:
            self.nu2 = np.asarray(fixed, dtype=np.float64)     # uploaded by the first sweep that uses it

    def _gaussian_noise(self):
        return True

    def _nu2_cells_model(self):
        """May nu2 be an array of known per-cell variances?  (The PG models' nu2 is the per-cell 1/omega they redraw
        every sweep.)"""
        return self._likelihood in (L.GAUSSIAN, L.CGAUSSIAN)

    def _likelihood_options(self):
        opts = super()._likelihood_options()
        if self._gaussian_noise():
            opts.update(nu2_a=self.nu2_a, nu2_b=self.nu2_b)
        return opts

    def _extra_init_mask(self):
        if not self._gaussian_noise():
            return super()._extra_init_mask()
        nu2_init, nu2_true = self._nu2_args
        self.sample_nu2 = nu2_true is None
        return L.INIT_NU2 if (nu2_init is None and nu2_true is None) else 0

    def _after_base_init(self):
        if not self._gaussian_noise():
            return super()._after_base_init()
        nu2_init, nu2_true = self._nu2_args
        fixed = nu2_true if nu2_true is not None else nu2_init
        if fixed is None or (self._nu2_cells_model() and np.size(fixed) != 1):
            return
        self._engine.set('nu2', [fixed])

    def _scalar_names(self):
        names = super()._scalar_names()
        if not self._gaussian_noise():
            return names
        return names if self._nu2_per_cell() is not None else names + ['nu2']

    def _nu2_per_cell(self):
        if not (self._gaussian_noise() and self._nu2_cells_model()):
            return super()._nu2_per_cell()
        nu2 = getattr(self, 'nu2', None)
        if np.size(nu2) == 1:
            return None
        nu2 = np.asarray(nu2, dtype=np.float64)
        shape = (self.nrows, self.ncols, self.ndepth)
        if nu2.shape != shape:
            raise ValueError('nu2 must be a scalar or an array of per-cell variances of shape %r, got %r'
                             % (shape, nu2.shape))
        return None if self.sample_nu2 else nu2

    def _push_state(self):
        super()._push_state()
        if not self._gaussian_noise():
            return
        cells = self._nu2_per_cell()
        # re-uploaded only when the variances changed (same rule as the data, see _fingerprint)
        key = None if cells is None else self._fingerprint(cells, getattr(self, '_full_check', False))
        if key != self._nu2_key:
            self._nu2_key = None      # the engine is in scalar mode after a refused upload
            self._engine.set_nu2_cells(None if cells is None else self._local_rows(cells))
            self._nu2_key = key

    def _init_nu2(self):
        self._engine.init_state(L.INIT_NU2)
        self.nu2 = self._engine.get_scalar('nu2')

    def _finish_results(self, results):
        results = super()._finish_results(results)
        if not self._gaussian_noise():
            return results
        nu2 = results.pop('_nu2_scalar')
        cells = self._nu2_per_cell()
        if cells is not None:
            nu2 = np.broadcast_to(cells, (nu2.shape[0],) + cells.shape)
        results['nu2'] = nu2
        return results

    def _inferred_variables(self, var_map):
        super()._inferred_variables(var_map)
        if self._gaussian_noise():
            var_map['nu2'] = self.nu2


class GaussianBayesianTensorFiltering(_GaussianNoise, BayesianTensorFiltering):
    """factor.py:286-423.  ``nu2`` is a scalar or an [N, M, T] array of known per-cell variances (see _GaussianNoise):
    with the array the W and V steps weight every cell by cnt / nu2[n, m, t]."""
    _likelihood = L.GAUSSIAN

    def _upload(self, data):
        Y = np.asarray(data)
        assert len(Y.shape) == 3 or len(Y.shape) == 4, 'Observations must be 3- or 4-tensor.'
        key = self._fingerprint(data, getattr(self, '_full_check', False))
        self._data_nbytes = int(np.asarray(data).nbytes)
        if key != self._data_key:
            self._engine.set_data_gaussian(self._local_rows(Y))
            self._data_key = key


class BinomialBayesianTensorFiltering(GaussianBayesianTensorFiltering):
    """factor.py:425-460: Polya-Gamma augmentation; ``nu2 = 1/omega`` per cell."""
    _likelihood = L.BINOMIAL
    # results['nu2'] is [nsamples, N, M, T] in the reference (factor.py:421-423 via 433);
    # above this many bytes it is skipped with a warning (SURVEY.md Q10)
    max_nu2_result_bytes = 2 << 30

    def __init__(self, nrows, ncols, ndepth, pg_seed=42, **kwargs):
        self.pg_seed = pg_seed
        kwargs.setdefault('nu2_init', 1.0)      # the Gaussian nu2 scalar is unused on the PG paths
        super().__init__(nrows, ncols, ndepth, **kwargs)
        self.sample_nu2 = True

    def _scalar_names(self):
        return ['sigma2', 'lam2', 'lam2_a']

    @property
    def nu2(self):
        with np.errstate(divide='ignore'):
            return 1.0 / self._engine.get('omega')

    @nu2.setter
    def nu2(self, value):
        # the per-cell variances live on the device as omega = 1 / nu2 (redrawn at the start of every resample,
        # factor.py:447-460, so like in the reference an assignment only lasts until the next sweep)
        v = np.asarray(value, dtype=np.float64)
        shape = (self._engine.nloc, self.ncols, self.ndepth)
        if v.shape != shape:
            raise ValueError('nu2 of a Polya-Gamma model is the per-cell tensor 1/omega of shape %r, got %r'
                             % (shape, v.shape))
        with np.errstate(divide='ignore'):
            self._engine.set('omega', np.where(np.isfinite(v) & (v > 0), 1.0 / v, 0.0))

    def _init_nu2(self):
        pass   # factor.py:433: the PG models start from nu2 = 0 and redraw it at the top of every resample

    def _upload(self, data):
        Y, N = data
        full = getattr(self, '_full_check', False)
        key = (self._fingerprint(Y, full), self._fingerprint(N, full))
        self._data_nbytes = int(np.asarray(Y).nbytes)
        if key != self._data_key:
            self._engine.set_data_binomial(self._local_rows(np.asarray(Y)), self._local_rows(np.asarray(N)))
            self._data_key = key

    def _alloc_results(self, nsamples):
        res = super()._alloc_results(nsamples)
        nbytes = nsamples * self._engine.nloc * self.ncols * self.ndepth * 8
        if nbytes <= self.max_nu2_result_bytes:
            res['_omega'] = np.empty((nsamples, self._engine.nloc, self.ncols, self.ndepth))
        else:
            warnings.warn('results["nu2"] would need %.1f GB; skipped (raise max_nu2_result_bytes to keep it)'
                          % (nbytes / 2.0 ** 30))
        return res

    def _result_buffers(self, results):
        outs = super()._result_buffers(results)
        if '_omega' in results:
            outs['omega'] = results['_omega']
        return outs

    def _finish_results(self, results):
        results = BayesianTensorFiltering._finish_results(self, results)
        results.pop('_nu2_scalar')
        if '_omega' in results:
            with np.errstate(divide='ignore'):
                results['nu2'] = 1.0 / results.pop('_omega')
        return results


class NegativeBinomialBayesianTensorFiltering(BinomialBayesianTensorFiltering):
    """factor.py:463-563: dispersion R by random-walk MH, then the Binomial sweep."""
    _likelihood = L.NEGBINOMIAL

    def __init__(self, nrows, ncols, ndepth, R_true=None, R_init=None, nmetropolis=30, rpropstdev=0.1,
                 rstdev=1, rdims=(0, 1, 2), **kwargs):
        self.nmetropolis, self.rpropstdev, self.rstdev = nmetropolis, rpropstdev, rstdev
        self._rdims_user = tuple(sorted(rdims)) if rdims is not None else ()
        self.rdims = [3] + list(self._rdims_user)[::-1]
        self._R_args = (R_true, R_init)
        self.sample_R = R_true is None
        super().__init__(nrows, ncols, ndepth, **kwargs)

    def _likelihood_options(self):
        opts = super()._likelihood_options()
        mask = 0
        for d in self._rdims_user:
            mask |= 1 << d
        opts.update(nmetropolis=int(self.nmetropolis), rpropstdev=float(self.rpropstdev),
                    rstdev=float(self.rstdev), rdims_mask=mask)
        return opts

    def _extra_init_mask(self):
        R_true, R_init = self._R_args
        self.sample_nu2 = True
        return L.INIT_R if (R_true is None and R_init is None) else 0

    def _after_base_init(self):
        R_true, R_init = self._R_args
        fixed = R_true if R_true is not None else R_init
        if fixed is not None:
            shape = self._engine.state_shape('R')
            self._engine.set('R', np.broadcast_to(np.asarray(fixed, dtype=float), shape))

    def _push_state(self):
        super()._push_state()
        self._engine.set('R', np.broadcast_to(np.asarray(self.R, dtype=float), self._engine.state_shape('R')))

    def _pull_state(self):
        super()._pull_state()
        self.R = self._engine.get('R')

    @property
    def N(self):
        return self._engine.get('Ntrials')

    def _upload(self, data):
        Y = np.asarray(data)
        key = self._fingerprint(data, getattr(self, '_full_check', False))
        self._data_nbytes = int(np.asarray(data).nbytes)
        if key != self._data_key:
            self._engine.set_data_negbin(self._local_rows(Y))
            self._data_key = key

    def _alloc_results(self, nsamples):
        res = super()._alloc_results(nsamples)
        res['R'] = np.empty((nsamples,) + tuple(self._engine.state_shape('R')))
        return res

    def _result_buffers(self, results):
        outs = super()._result_buffers(results)
        outs['R'] = results['R']
        return outs

    def _inferred_variables(self, var_map):
        super()._inferred_variables(var_map)
        var_map['R'] = self.R
