"""Thin numpy-facing wrapper of the C engine handle (one engine = one GPU)."""
import ctypes as C
import weakref
import numpy as np

from . import _lib as L


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)


PINNED_LOG = []      # (nbytes, how) for every pinned_empty call: 'alloc', 'registered' or 'pageable'


def pinned_empty(shape):
    """float64 array in page-locked host memory: a fresh pinned allocation, else a pageable
    array page-locked in place, else (logged in PINNED_LOG) plain pageable memory."""
    lib = L.load()
    n = int(np.prod(shape)) if len(shape) else 1
    nbytes = max(n, 1) * 8
    p = lib.btf_host_alloc(nbytes)
    if p:
        buf = (C.c_double * max(n, 1)).from_address(p)
        arr = np.frombuffer(buf, dtype=np.float64, count=n).reshape(shape)
        weakref.finalize(buf, lib.btf_host_free, p)
        PINNED_LOG.append((nbytes, 'alloc'))
        return arr
    arr = np.empty(shape, dtype=np.float64)
    if arr.size and lib.btf_host_register(C.c_void_p(arr.ctypes.data), arr.nbytes) == 0:
        weakref.finalize(arr, lib.btf_host_unregister, C.c_void_p(arr.ctypes.data))
        PINNED_LOG.append((nbytes, 'registered'))
    else:
        PINNED_LOG.append((nbytes, 'pageable'))
    return arr


class Engine(object):
    """Owns a ``btf_engine*``.  All arrays crossing this boundary are float64."""

    def __init__(self, nrows, ncols, ndepth, nembeds=5, tf_order=2, likelihood=L.GAUSSIAN, **opts):
        self.lib = L.load()
        cfg = L.Config()
        self.lib.btf_config_default(C.byref(cfg))
        cfg.nrows, cfg.ncols, cfg.ndepth = int(nrows), int(ncols), int(ndepth)
        cfg.nembeds, cfg.tf_order, cfg.likelihood = int(nembeds), int(tf_order), int(likelihood)
        names = set(f[0] for f in L.Config._fields_)
        for k, v in opts.items():
            if k not in names:
                raise TypeError('unknown engine option %r' % k)
            setattr(cfg, k, v)
        self.cfg = cfg
        h = C.c_void_p(0)
        L.check(self.lib.btf_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self._finalizer = weakref.finalize(self, self.lib.btf_destroy, h)
        self.N, self.M, self.T, self.K = cfg.nrows, cfg.ncols, cfg.ndepth, cfg.nembeds
        self.RD = self.lib.btf_delta_rows(h)
        ws = max(1, cfg.world_size)
        self.nloc = (cfg.row_end - cfg.row_begin) if ws > 1 else cfg.nrows
        self.Mloc = (cfg.col_end - cfg.col_begin) if ws > 1 else cfg.ncols
        self.likelihood = cfg.likelihood
        self._keep = []

    def close(self):
        self._finalizer()

    # ---- shapes
    def state_shape(self, name):
        N, M, T, K, RD = self.N, self.M, self.T, self.K, self.RD
        if name == 'W':
            return (N, K)
        if name == 'V':
            return (M, T, K)
        if name in ('Tau2', 'Tau2_a', 'Tau2_b', 'Tau2_c'):
            return (M, RD)
        if name in ('omega', 'Ntrials', 'kappa'):
            return (self.nloc, M, T)
        if name == 'Delta':
            return (RD, T)
        if name == 'R':
            m = self.cfg.rdims_mask
            return (1 if m & 1 else N, 1 if m & 2 else M, 1 if m & 4 else T)
        return (1,)

    # ---- data
    def set_data_gaussian(self, Y):
        Y = np.asarray(Y)
        if Y.ndim == 3:
            Y = Y[..., None]
        if Y.ndim != 4 or Y.shape[:3] != (self.nloc, self.M, self.T):
            raise ValueError('Observations must be a [%d,%d,%d(,R)] tensor, got %s'
                             % (self.nloc, self.M, self.T, Y.shape))
        Y = _f64(Y)
        L.check(self.lib.btf_set_data_gaussian(self._h, _ptr(Y), Y.shape[3]))

    def set_data_gaussian_device(self, dev_ptr, nreps):
        L.check(self.lib.btf_set_data_gaussian(self._h, C.c_void_p(int(dev_ptr)), int(nreps)))

    def set_data_gaussian_rows_device(self, dev_ptr, row0, nrows, nreps, reset):
        """Streaming form: a device-resident piece [nrows, M, T, nreps] of the local shard."""
        L.check(self.lib.btf_set_data_gaussian_rows(self._h, C.c_void_p(int(dev_ptr)), int(row0), int(nrows),
                                                    int(nreps), 1 if reset else 0))

    def set_data_binomial(self, Y, Nt):
        """Successes and trials [Nloc, M, T] of a Binomial or constrained Binomial engine (NaN = missing)."""
        Y, Nt = _f64(Y), _f64(Nt)
        if Y.shape != (self.nloc, self.M, self.T) or Nt.shape != Y.shape:
            raise ValueError('Binomial data must be two [%d,%d,%d] tensors' % (self.nloc, self.M, self.T))
        L.check(self.lib.btf_set_data_binomial(self._h, _ptr(Y), _ptr(Nt)))

    def set_data_negbin(self, Y):
        Y = np.asarray(Y)
        if Y.ndim == 3:
            Y = Y[..., None]
        if Y.ndim != 4 or Y.shape[:3] != (self.nloc, self.M, self.T):
            raise ValueError('Counts must be a [%d,%d,%d(,R)] tensor' % (self.nloc, self.M, self.T))
        Y = _f64(Y)
        L.check(self.lib.btf_set_data_negbin(self._h, _ptr(Y), Y.shape[3]))

    def set_nu2_cells(self, nu2):
        """Known per-cell noise variances [Nloc, M, T] of a Gaussian or constrained Gaussian engine (``None``: back to
        the scalar nu2)."""
        a = None
        if nu2 is not None:
            a = _f64(nu2)
            if a.shape != (self.nloc, self.M, self.T):
                raise ValueError('nu2 must be a [%d,%d,%d] tensor, got %s' % (self.nloc, self.M, self.T, a.shape))
        L.check(self.lib.btf_set_nu2_cells(self._h, _ptr(a)))

    def set_data_poisson(self, Y):
        """Counts [Nloc, M, T(, R)] of a Poisson engine (NaN = missing)."""
        Y = np.asarray(Y)
        if Y.ndim == 3:
            Y = Y[..., None]
        if Y.ndim != 4 or Y.shape[:3] != (self.nloc, self.M, self.T):
            raise ValueError('Counts must be a [%d,%d,%d(,R)] tensor, got %s' % (self.nloc, self.M, self.T, Y.shape))
        Y = _f64(Y)
        L.check(self.lib.btf_set_data_poisson(self._h, _ptr(Y), Y.shape[3]))

    def set_gass(self, A, C, grid_fine, grid_coarse, rowcons=None):
        """Constraints A [J, T] tau >= C [J] on every cell's depth profile, optional row constraints [nrc, K + 1] on W,
        and the fine / coarse angle grids of the GASS steps (len(grid_coarse) = ngrid candidates)."""
        A = _f64(np.asarray(A, dtype=np.float64).reshape(-1, self.T))
        C = _f64(np.asarray(C, dtype=np.float64).reshape(-1))
        if C.shape[0] != A.shape[0]:
            raise ValueError('A has %d rows, C has %d entries' % (A.shape[0], C.shape[0]))
        R = None
        if rowcons is not None:
            R = _f64(np.asarray(rowcons, dtype=np.float64).reshape(-1, self.K + 1))
        gf, gc = _f64(grid_fine), _f64(grid_coarse)
        L.check(self.lib.btf_set_gass(self._h, _ptr(A), _ptr(C), A.shape[0], _ptr(R), 0 if R is None else R.shape[0],
                                      _ptr(gf), gf.size, _ptr(gc), gc.size))

    def set_ep(self, mu, sigma):
        """EP approximation N(mu, sigma^2) per cell [Nloc, M, T] of a constrained Poisson, Binomial or Gaussian engine
        (``None``: none)."""
        if mu is None:
            L.check(self.lib.btf_set_ep(self._h, C.c_void_p(0), C.c_void_p(0)))
            return
        shape = (self.nloc, self.M, self.T)
        m, s = _f64(mu), _f64(sigma)
        if m.shape != shape or s.shape != shape:
            raise ValueError('the EP approximation must be two %r tensors, got %r and %r' % (shape, m.shape, s.shape))
        L.check(self.lib.btf_set_ep(self._h, _ptr(m), _ptr(s)))

    # ---- state
    def set(self, name, value):
        a = _f64(np.asarray(value, dtype=np.float64).reshape(-1))
        L.check(self.lib.btf_set_state(self._h, name.encode(), _ptr(a), a.size))

    def get(self, name):
        shape = self.state_shape(name)
        a = np.empty(shape, dtype=np.float64)
        L.check(self.lib.btf_get_state(self._h, name.encode(), _ptr(a), a.size))
        return a

    def get_scalar(self, name):
        return float(self.get(name)[0])

    def set_sample_mask(self, mask):
        L.check(self.lib.btf_set_sample_mask(self._h, int(mask)))

    def init_state(self, mask):
        L.check(self.lib.btf_init_state(self._h, int(mask)))

    # ---- sampling
    def sweep(self, n=1):
        L.check(self.lib.btf_sweep(self._h, int(n)))

    def sweep_timed(self, n):
        ms = C.c_double(0.0)
        L.check(self.lib.btf_sweep_timed(self._h, int(n), C.byref(ms)))
        return ms.value

    def time_phases(self, n):
        out = (C.c_double * 16)()
        L.check(self.lib.btf_time_phases(self._h, int(n), out, 16))
        return dict(zip(L.PHASES, [out[i] for i in range(len(L.PHASES))]))

    def run_segment(self, nsweeps, first_save, nthin, sample_offset, W=None, V=None, Tau2=None,
                    scalars=None, R=None, omega=None):
        L.check(self.lib.btf_run_segment(self._h, int(nsweeps), int(first_save), int(nthin), int(sample_offset),
                                         _ptr(W), _ptr(V), _ptr(Tau2), _ptr(scalars), _ptr(R), _ptr(omega)))

    def track_mu_stats(self, on=True):
        L.check(self.lib.btf_mu_stats_track(self._h, 1 if on else 0))

    def mu_stats(self):
        """(mean, variance, count) of Mu over the samples saved since track_mu_stats(True)."""
        shape = (self.nloc, self.M, self.T)
        mean, var = np.empty(shape), np.empty(shape)
        cnt = C.c_int64(0)
        L.check(self.lib.btf_mu_stats_get(self._h, _ptr(mean), _ptr(var), C.byref(cnt)))
        return mean, var, int(cnt.value)

    # ---- held-out evaluation (btf_eval_*)
    def eval_set(self, slot, target, classes=None, nclasses=1, transform=0, loglik=0, cell_state=1,
                 auto_update=True, max_samples=1000):
        shape = (self.nloc, self.M, self.T)
        t = _f64(target)
        if t.shape != shape:
            raise ValueError('target must have the local shape %r, got %r' % (shape, t.shape))
        c = None
        if classes is not None:
            c = np.ascontiguousarray(classes, dtype=np.uint8)
            if c.shape != shape:
                raise ValueError('classes must have the local shape %r, got %r' % (shape, c.shape))
        L.check(self.lib.btf_eval_set(self._h, int(slot), _ptr(t), _ptr(c), int(nclasses), int(transform),
                                      int(loglik), int(cell_state), 1 if auto_update else 0, int(max_samples)))

    def eval_set_nu2(self, slot, nu2):
        """Per-cell variances [Nloc, M, T] for the Gaussian scores of an evaluator slot (``None``: the scalar nu2)."""
        a = None
        if nu2 is not None:
            a = _f64(nu2)
            if a.shape != (self.nloc, self.M, self.T):
                raise ValueError('nu2 must have the local shape %r, got %r' % ((self.nloc, self.M, self.T), a.shape))
        L.check(self.lib.btf_eval_set_nu2(self._h, int(slot), _ptr(a)))

    def eval_clear(self, slot):
        L.check(self.lib.btf_eval_clear(self._h, int(slot)))

    def eval_update(self, slot):
        L.check(self.lib.btf_eval_update(self._h, int(slot)))

    def eval_samples(self, slot, nclasses):
        cnt = C.c_int64(0)
        L.check(self.lib.btf_eval_samples(self._h, int(slot), C.c_void_p(0), C.byref(cnt)))
        out = np.empty((int(cnt.value), int(nclasses), 4), dtype=np.float64)
        L.check(self.lib.btf_eval_samples(self._h, int(slot), _ptr(out), C.byref(cnt)))
        return out

    def eval_summary(self, slot, nclasses, lo_pct, hi_pct, pred_lo=0.0, pred_hi=1.0, want_mean=False):
        out = np.empty((int(nclasses), 6), dtype=np.float64)
        mean = np.empty((self.nloc, self.M, self.T), dtype=np.float64) if want_mean else None
        L.check(self.lib.btf_eval_summary(self._h, int(slot), float(lo_pct), float(hi_pct), float(pred_lo),
                                          float(pred_hi), _ptr(out), _ptr(mean)))
        return (out, mean) if want_mean else out

    def synchronize(self):
        L.check(self.lib.btf_synchronize(self._h))

    # ---- parity hooks
    def inject(self, name, value):
        a = _f64(np.asarray(value, dtype=np.float64).reshape(-1))
        L.check(self.lib.btf_inject_noise(self._h, name.encode(), _ptr(a), a.size))

    def enable_diag(self, on=True):
        L.check(self.lib.btf_enable_diag(self._h, 1 if on else 0))

    def diag(self, name):
        N, M, T, K, RD = self.N, self.M, self.T, self.K, self.RD
        kd = (self.cfg.tf_order + 1) * K
        Lp = K * (K + 1) // 2
        shapes = {
            'W_Q': (N, K, K), 'W_L': (N, K, K), 'W_mean': (N, K), 'W_b': (N, K), 'V_mean': (M, T, K),
            'V_band': (self.Mloc, T * K, kd + 1), 'V_chol': (self.Mloc, T * K, kd + 1),
            'V_retries': (self.Mloc,), 'row_stats': (self.nloc, Lp + K), 'col_stats': (M * T, Lp + K),
            'gass_W': (N, 3), 'gass_V': (M, 3), 'nu2_rate': (3,), 'lam2_rate': (2,), 'info': (3,), 'i8_guard': (2,), 'i8_route': (2,),
        }
        a = np.empty(shapes[name], dtype=np.float64)
        L.check(self.lib.btf_get_diag(self._h, name.encode(), _ptr(a), a.size))
        return a

    @property
    def kernel_launches(self):
        return int(self.lib.btf_kernel_launches(self._h))

    # ---- multi GPU
    def nccl_init(self, unique_id):
        L.check(self.lib.btf_nccl_init(self._h, C.c_char_p(unique_id)))


def nccl_unique_id():
    lib = L.load()
    buf = C.create_string_buffer(128)
    L.check(lib.btf_nccl_unique_id(buf))
    return buf.raw


def fp64_peak(device=0, mode=1, iters=20000):
    return L.load().btf_fp64_peak(int(device), int(mode), int(iters))


def i8_peak(device=0, iters=4000):
    """Measured int8 tensor-core rate (Top/s) with operands resident in shared memory."""
    return L.load().btf_i8_peak(int(device), int(iters))


def hbm_copy_gbs(device=0, nbytes=1 << 30, iters=5):
    return L.load().btf_hbm_copy_gbs(int(device), int(nbytes), int(iters))


def pg_sample(b, z, seed=1, device=0):
    """omega[e] ~ PG(b[e], z[e]) from the device sampler."""
    b = _f64(np.broadcast_to(np.asarray(b, dtype=np.float64), np.broadcast(b, z).shape).ravel())
    z = _f64(np.broadcast_to(np.asarray(z, dtype=np.float64), b.shape).ravel())
    out = np.empty_like(b)
    L.check(L.load().btf_pg_sample(int(device), _ptr(b), _ptr(z), _ptr(out), b.size, int(seed)))
    return out


def rng_sample(kind, n, param=0.0, seed=1, device=0):
    """Raw variates of the device Philox generator: 'normal', 'gamma', 'exponential', 'uniform'."""
    code = {'normal': 0, 'gamma': 1, 'exponential': 2, 'uniform': 3}[kind]
    out = np.empty(int(n), dtype=np.float64)
    L.check(L.load().btf_rng_sample(int(device), code, float(param), _ptr(out), out.size, int(seed)))
    return out
