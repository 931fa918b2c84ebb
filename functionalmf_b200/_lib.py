"""ctypes binding of libbtf_b200.so (C ABI declared in include/btf_b200.h).

There is NO CPU fallback: if the CUDA library is missing or cannot be loaded,
importing the sampler classes still works (so host-only helpers and CPU tests can
run) but creating an engine raises ``BTFLibraryError``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# BTF_B200_LIB: developer hook for instrumented builds of the same library (tools/band_profile.py)
LIB_PATH = os.environ.get('BTF_B200_LIB') or os.path.join(_HERE, 'libbtf_b200.so')

BTF_OK, BTF_EINVAL, BTF_ECUDA, BTF_ENOTPD, BTF_ESTATE, BTF_ENCCL = 0, -1, -2, -3, -4, -5
GAUSSIAN, BINOMIAL, NEGBINOMIAL, POISSON, CBINOMIAL, CGAUSSIAN = 0, 1, 2, 3, 4, 5   # C*: constrained Binomial / Gaussian (GASS)
SAMPLE_NU2, SAMPLE_SIGMA2, SAMPLE_TAU2, SAMPLE_LAM2, SAMPLE_W, SAMPLE_V, SAMPLE_R = 1, 2, 4, 8, 16, 32, 64
SAMPLE_ALL = 127
I8_ROUTE_FUSED, I8_ROUTE_SPLITK = 2, 3     # btf_get_diag("i8_route")
INIT_SIGMA2, INIT_LAM2, INIT_NU2, INIT_TAU2, INIT_W, INIT_V, INIT_R = 1, 2, 4, 8, 16, 32, 64
PHASES = ['nu2_or_pg', 'sigma2', 'tau2', 'lam2', 'row_stats', 'row_solve', 'col_stats', 'band_solve', 'comm',
          # sub-phases of row_stats / col_stats on the integer-tensor-core path (0 when it is off)
          'row_i8gemm', 'row_linear', 'col_i8gemm', 'col_linear']


class BTFLibraryError(RuntimeError):
    pass


class BTFError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, 'btf_b200 error %d: %s' % (code, msg))
        self.code = code


class NotPositiveDefiniteError(BTFError, ArithmeticError):
    """A Cholesky factorisation failed (np.linalg.LinAlgError in the reference)."""


class Config(C.Structure):
    """struct btf_config (include/btf_b200.h)."""
    _fields_ = [
        ('nrows', C.c_int32), ('ncols', C.c_int32), ('ndepth', C.c_int32),
        ('nembeds', C.c_int32), ('tf_order', C.c_int32), ('likelihood', C.c_int32),
        ('sigma2_a', C.c_double), ('sigma2_b', C.c_double),
        ('nu2_a', C.c_double), ('nu2_b', C.c_double), ('stability', C.c_double),
        ('force_psd', C.c_int32), ('force_psd_attempts', C.c_int32), ('force_psd_eps', C.c_double),
        ('ref_compat_lam2', C.c_int32), ('sample_mask', C.c_int32),
        ('seed', C.c_uint64), ('device', C.c_int32),
        ('nmetropolis', C.c_int32), ('rpropstdev', C.c_double), ('rstdev', C.c_double),
        ('rdims_mask', C.c_int32),
        ('row_begin', C.c_int32), ('row_end', C.c_int32), ('col_begin', C.c_int32), ('col_end', C.c_int32),
        ('world_size', C.c_int32), ('rank', C.c_int32),
        ('resid_direct', C.c_int32), ('use_graph', C.c_int32),
        ('stats_splits_row', C.c_int32), ('stats_splits_col', C.c_int32),
        ('clip_prior_precision', C.c_int32),
    ]


# every symbol include/btf_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_D = C.POINTER(C.c_double)
SIGNATURES = {
    'btf_config_default': (None, [C.POINTER(Config)]),
    'btf_create': (C.c_int, [C.POINTER(Config), C.POINTER(_P)]),
    'btf_destroy': (None, [_P]),
    'btf_last_error': (C.c_char_p, []),
    'btf_set_data_gaussian': (C.c_int, [_P, _P, C.c_int32]),
    'btf_set_data_gaussian_rows': (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    'btf_set_data_binomial': (C.c_int, [_P, _P, _P]),
    'btf_set_data_negbin': (C.c_int, [_P, _P, C.c_int32]),
    'btf_set_nu2_cells': (C.c_int, [_P, _P]),
    'btf_set_data_poisson': (C.c_int, [_P, _P, C.c_int32]),
    'btf_set_gass': (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_int32, _P, C.c_int32, _P, C.c_int32]),
    'btf_set_ep': (C.c_int, [_P, _P, _P]),
    'btf_set_state': (C.c_int, [_P, C.c_char_p, _P, C.c_size_t]),
    'btf_get_state': (C.c_int, [_P, C.c_char_p, _P, C.c_size_t]),
    'btf_delta_rows': (C.c_int, [_P]),
    'btf_set_sample_mask': (C.c_int, [_P, C.c_int32]),
    'btf_sweep': (C.c_int, [_P, C.c_int32]),
    'btf_run': (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P]),
    'btf_run_segment': (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int64, _P, _P, _P, _P, _P, _P]),
    'btf_synchronize': (C.c_int, [_P]),
    'btf_init_state': (C.c_int, [_P, C.c_int32]),
    'btf_mu_stats_track': (C.c_int, [_P, C.c_int32]),
    'btf_mu_stats_get': (C.c_int, [_P, _P, _P, C.POINTER(C.c_int64)]),
    'btf_eval_set': (C.c_int, [_P, C.c_int32, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64]),
    'btf_eval_set_nu2': (C.c_int, [_P, C.c_int32, _P]),
    'btf_eval_clear': (C.c_int, [_P, C.c_int32]),
    'btf_eval_update': (C.c_int, [_P, C.c_int32]),
    'btf_eval_samples': (C.c_int, [_P, C.c_int32, _P, C.POINTER(C.c_int64)]),
    'btf_eval_summary': (C.c_int, [_P, C.c_int32, C.c_double, C.c_double, C.c_double, C.c_double, _P, _P]),
    'btf_host_alloc': (_P, [C.c_size_t]),
    'btf_host_free': (None, [_P]),
    'btf_host_register': (C.c_int, [_P, C.c_size_t]),
    'btf_host_unregister': (C.c_int, [_P]),
    'btf_sweep_timed': (C.c_int, [_P, C.c_int32, _D]),
    'btf_inject_noise': (C.c_int, [_P, C.c_char_p, _P, C.c_size_t]),
    'btf_enable_diag': (C.c_int, [_P, C.c_int32]),
    'btf_get_diag': (C.c_int, [_P, C.c_char_p, _P, C.c_size_t]),
    'btf_kernel_launches': (C.c_int64, [_P]),
    'btf_time_phases': (C.c_int, [_P, C.c_int32, _D, C.c_int32]),
    'btf_fp64_peak': (C.c_double, [C.c_int32, C.c_int32, C.c_int32]),
    'btf_hbm_copy_gbs': (C.c_double, [C.c_int32, C.c_size_t, C.c_int32]),
    'btf_i8_peak': (C.c_double, [C.c_int32, C.c_int32]),
    'btf_pg_sample': (C.c_int, [C.c_int32, _P, _P, _P, C.c_int64, C.c_uint64]),
    'btf_rng_sample': (C.c_int, [C.c_int32, C.c_int32, C.c_double, _P, C.c_int64, C.c_uint64]),
    'btf_nccl_unique_id': (C.c_int, [C.c_char_p]),
    'btf_nccl_init': (C.c_int, [_P, C.c_char_p]),
}

_lib = None


def load():
    """Load (once) and return the ctypes handle; raises BTFLibraryError if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BTFLibraryError(
            'libbtf_b200.so not found at %s -- build it with `python -c "import __graft_entry__ as g; g.build()"` '
            '(functionalmf_b200/csrc/build.sh); there is no CPU fallback' % LIB_PATH)
    try:
        lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    except OSError as exc:
        raise BTFLibraryError('cannot load %s: %s (there is no CPU fallback)' % (LIB_PATH, exc))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc == BTF_OK:
        return
    msg = load().btf_last_error().decode('utf-8', 'replace')
    if rc == BTF_ENOTPD:
        raise NotPositiveDefiniteError(rc, msg)
    raise BTFError(rc, msg)
