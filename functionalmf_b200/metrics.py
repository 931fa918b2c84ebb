"""Held-out scoring of a chain on the device (SURVEY.md 8f row 3).

The reference's application scripts keep every saved (W, V) sample, rebuild the
whole ``[nsamples, N, M, T]`` surface with ``np.einsum`` and score it with numpy
(politics/benchmark.py:153-180, flutrends/benchmark.py:48-75 and 129-143,
examples/poisson_tensor_filtering.py:20-23 and 165-173).  ``HeldOutEvaluator``
produces the same numbers from one extra pass over the resident factors per saved
sample (``btf_eval_*`` in include/btf_b200.h), so neither the samples nor the
surface ever have to exist:

    ev = HeldOutEvaluator(model, Y, train=Y_train, transform='nb_mean', loglik='poisson')
    results = model.run_gibbs(Y_train, nburn=..., nsamples=...)
    ev.rmse(), ev.mae(), ev.loglik()          # mean over samples of the per-sample score, per class
    ev.rmse_of_mean(), ev.mae_of_mean()       # score of the posterior-mean surface
    ev.coverage(95)                           # target inside the central 95 % np.percentile band
    ev.predictive_coverage(95)                # Gaussian posterior-predictive band (flutrends)

Classes: with ``train=`` the cells are split like the scripts do — class 0
"in_sample" = observed in both, class 1 "held_out" = observed in ``target`` but NaN
in ``train``; cells that are NaN in ``target`` are not scored.  ``classes=`` gives an
explicit uint8 array instead (values >= nclasses are not scored).
"""
import numpy as np

TRANSFORMS = {'identity': 0, 'ilogit': 1, 'nb_mean': 2}
LOGLIKS = {None: 0, 'none': 0, 'gaussian': 1, 'poisson': 2}
IGNORE = 255


def heldout_classes(target, train):
    """uint8 classes: 0 in-sample, 1 held out, 255 missing (politics/benchmark.py:164-166)."""
    target, train = np.asarray(target), np.asarray(train)
    is_missing = np.isnan(target)
    is_held_out = (~is_missing) & np.isnan(train)
    cls = np.full(target.shape, IGNORE, dtype=np.uint8)
    cls[(~is_missing) & (~is_held_out)] = 0
    cls[is_held_out] = 1
    return cls


class HeldOutEvaluator(object):
    def __init__(self, model, target, train=None, classes=None, class_names=None, transform='identity',
                 loglik=None, cell_state=True, predictive=False, max_samples=None, slot=None):
        self.model = model
        eng = model._engine
        target = np.asarray(target, dtype=np.float64)
        if target.ndim != 3:
            raise ValueError('target must be [nrows, ncols, ndepth]')
        if train is not None and classes is not None:
            raise ValueError('give either train= or classes=')
        if train is not None:
            train = np.asarray(train, dtype=np.float64)
            if train.ndim == 4:    # replicated observations: held out = no replicate observed
                train = np.where(np.isnan(train).all(axis=-1), np.nan, 0.0)
            classes = heldout_classes(target, train)
            class_names = class_names or ('in_sample', 'held_out')
        if classes is None:
            class_names = class_names or ('all',)
        else:
            classes = np.asarray(classes, dtype=np.uint8)
            if class_names is None:
                class_names = tuple('class%d' % c for c in range(int(classes[classes != IGNORE].max(initial=0)) + 1))
        self.class_names = tuple(class_names)
        self.nclasses = len(self.class_names)
        self.transform, self.loglik_kind = transform, loglik
        used = getattr(model, '_evaluators', None)
        if used is None:
            used = model._evaluators = {}
        if slot is None:
            free = [s for s in range(4) if s not in used]
            if not free:
                raise RuntimeError('an engine holds at most 4 evaluators; close() one first')
            slot = free[0]
        self.slot = slot
        self._cell_state = (2 if predictive else 1) if (cell_state or predictive) else 0
        self._max_samples = max_samples
        self._target = model._local_rows(target)
        self._classes = None if classes is None else model._local_rows(classes)
        self._armed = False
        if max_samples is not None:
            self._arm(max_samples)
        used[slot] = self          # registered only once construction succeeded

    # the engine buffers are sized when the chain length is known (run_gibbs arms the evaluator)
    def _arm(self, nsamples):
        self.model._engine.eval_set(self.slot, self._target, self._classes, self.nclasses,
                                    TRANSFORMS[self.transform], LOGLIKS[self.loglik_kind], self._cell_state,
                                    auto_update=True, max_samples=max(int(nsamples), 1))
        cells = self.model._nu2_per_cell()
        if cells is not None:        # known per-cell variances: the Gaussian scores use them, not the scalar nu2
            self.model._engine.eval_set_nu2(self.slot, self.model._local_rows(cells))
        self._armed = True

    def update(self):
        """Score the model's current state as one more sample (for ``resample`` loops)."""
        if not self._armed:
            self._arm(self._max_samples or 1000)
        self.model._push_state()
        self.model._engine.eval_update(self.slot)

    def close(self):
        self.model._engine.eval_clear(self.slot)
        self.model._evaluators.pop(self.slot, None)
        self._armed = False

    # ---- sums over ranks
    def _allreduce(self, a):
        shard = getattr(self.model, '_shard', None)
        if shard is not None and shard.world_size > 1:
            import torch
            import torch.distributed as dist
            t = torch.from_numpy(np.ascontiguousarray(a))
            if dist.get_backend() == 'nccl':
                t = t.cuda()
            dist.all_reduce(t)
            a = t.cpu().numpy()
        return a

    def per_sample(self):
        """[nsamples, nclasses, 4] = n, sum (y-mu)^2, sum |y-mu|, sum loglik for every scored sample."""
        return self._allreduce(self.model._engine.eval_samples(self.slot, self.nclasses))

    def _named(self, values):
        return {name: float(v) for name, v in zip(self.class_names, values)}

    def rmse(self):
        """Mean over samples of sqrt(mean_cells (y - mu_s)^2) (politics/benchmark.py:168-170)."""
        s = self.per_sample()
        return self._named(np.sqrt(s[:, :, 1] / s[:, :, 0]).mean(axis=0))

    def mae(self):
        s = self.per_sample()
        return self._named((s[:, :, 2] / s[:, :, 0]).mean(axis=0))

    def loglik(self):
        """Mean over samples of the mean log-likelihood per cell (politics/benchmark.py:176-178)."""
        s = self.per_sample()
        return self._named((s[:, :, 3] / s[:, :, 0]).mean(axis=0))

    def _summary(self, lo_pct=2.5, hi_pct=97.5, pred_lo=0.025, pred_hi=0.975):
        return self._allreduce(self.model._engine.eval_summary(self.slot, self.nclasses, lo_pct, hi_pct,
                                                               pred_lo, pred_hi))

    def posterior_mean(self):
        """Posterior mean of the transformed surface, local rows [Nloc, M, T]."""
        return self.model._engine.eval_summary(self.slot, self.nclasses, 2.5, 97.5, want_mean=True)[1]

    def rmse_of_mean(self):
        """sqrt(mean (y - E[mu])^2) (flutrends/benchmark.py:136-138, utils.py:109-110)."""
        s = self._summary()
        return self._named(np.sqrt(s[:, 1] / s[:, 0]))

    def mae_of_mean(self):
        s = self._summary()
        return self._named(s[:, 2] / s[:, 0])

    def nll_of_mean(self):
        """-sum loglik(y | E[mu]) (examples/poisson_tensor_filtering.py:168)."""
        s = self._summary()
        return self._named(-s[:, 3])

    def coverage(self, interval=95):
        """Percentage of targets inside the central ``interval`` % percentile band of the samples
        (coverage_at, examples/poisson_tensor_filtering.py:20-23)."""
        lo = (100 - interval) / 2
        s = self._summary(lo, lo + interval)
        return self._named(s[:, 4] / s[:, 0] * 100)

    def predictive_coverage(self, interval=95):
        """Percentage of targets inside the central band of the Gaussian posterior predictive
        (flutrends/benchmark.py:68-75 draws it by Monte Carlo; this is its exact mixture limit)."""
        if self._cell_state < 2:
            raise RuntimeError('construct the evaluator with predictive=True')
        lo = (100 - interval) / 200
        s = self._summary(pred_lo=lo, pred_hi=1 - lo)
        return self._named(s[:, 5] / s[:, 0] * 100)
