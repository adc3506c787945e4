"""ctypes binding of libgladsgp_b200.so (the C ABI in include/gladsgp_b200.h).

There is no CPU fallback: every compute entry point raises if the library or a CUDA device is
missing.  Device buffers are torch tensors (used for memory and streams only).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libgladsgp_b200.so')
_lib = None


class GgpError(RuntimeError):
    pass


class McmcArgs(C.Structure):
    _fields_ = [
        ('m', C.c_int), ('d', C.c_int), ('pu', C.c_int), ('n_chains', C.c_int), ('n_steps', C.c_int),
        ('do_propMH', C.c_int), ('replay', C.c_int), ('init_sigwl', C.c_int), ('per_chain_data', C.c_int),
        ('X', C.c_void_p), ('W', C.c_void_p), ('lamsim', C.c_void_p),
        ('prior_kind', C.c_void_p), ('prior_a', C.c_void_p), ('prior_b', C.c_void_p),
        ('lo', C.c_void_p), ('hi', C.c_void_p), ('prop_kind', C.c_void_p), ('fixed', C.c_void_p),
        ('step', C.c_void_p), ('step_stride_t', C.c_longlong), ('step_stride_c', C.c_longlong),
        ('theta', C.c_void_p), ('sigwl', C.c_void_p),
        ('uniforms', C.c_void_p), ('n_uniform', C.c_longlong), ('upos', C.c_void_p),
        ('r_cand', C.c_void_p), ('r_logacorr', C.c_void_p), ('r_logu', C.c_void_p), ('r_valid', C.c_void_p),
        ('draws', C.c_void_p), ('lp_draws', C.c_void_p), ('accepted', C.c_void_p),
        ('workspace', C.c_void_p), ('workspace_bytes', C.c_size_t),
        ('eval_count', C.c_void_p), ('kernel_ms', C.c_void_p),
        ('pc_begin', C.c_int), ('pc_count', C.c_int), ('step_index', C.c_int), ('reserved0', C.c_int),
        ('xchg', C.c_void_p),
    ]


_I, _LL, _P, _D, _F = C.c_int, C.c_longlong, C.c_void_p, C.c_double, C.c_float

# name -> (restype, argtypes); mirrors include/gladsgp_b200.h one to one
SIGNATURES = {
    'ggp_version': (_I, []),
    'ggp_last_error_string': (C.c_char_p, []),
    'ggp_device_info': (_I, [C.POINTER(_I), C.POINTER(_I), C.POINTER(_I), C.POINTER(_LL)]),
    'ggp_cov_build_f64': (_I, [_P, _I, _I, _P, _P, _P, _I, _P, _P]),
    'ggp_cross_cov_f64': (_I, [_P, _I, _P, _I, _I, _P, _P, _I, _P, _P]),
    'ggp_debug_exp_neg_f64': (_I, [_P, _P, _I, _P]),
    'ggp_factor_doubles': (_LL, [_I]),
    'ggp_padded_m': (_I, [_I]),
    'ggp_set_lookahead': (_I, [_I]),
    'ggp_loglik_batched_f64': (_I, [_P, _I, _I, _P, _LL, _P, _P, _P, _I, _P, _P, _P, _P, _P]),
    'ggp_factor_unpack_f64': (_I, [_P, _I, _I, _P, _P]),
    'ggp_sizeof_mcmc_args': (_I, []),
    'ggp_mcmc_workspace_bytes': (_LL, [_I, _I, _I, _I]),
    'ggp_mcmc_run_f64': (_I, [C.POINTER(McmcArgs), _P]),
    'ggp_mcmc_plan_f64': (_I, [C.POINTER(McmcArgs), _I, _P]),
    'ggp_mcmc_close_f64': (_I, [C.POINTER(McmcArgs), _I, _I, _P]),
    'ggp_predict_workspace_bytes': (_LL, [_I, _I, _I]),
    'ggp_predict_f64': (_I, [_P, _I, _I, _P, _P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _LL, _P]),
    'ggp_pred_cov_f64': (_I, [_P, _I, _I, _P, _P, _P, _P, _I, _I, _P, _P]),
    'ggp_chol_draw_workspace_bytes': (_LL, [_I, _I]),
    'ggp_chol_draw_f64': (_I, [_P, _I, _I, _P, _P, _P, _P, _LL, _P]),
    'ggp_xval_workspace_bytes': (_LL, [_I, _I, _I]),
    'ggp_xval_solve_f64': (_I, [_P, _P, _I, _I, _P, _I, _P, _P, _P, _P, _LL, _P]),
    'ggp_reconstruct_f32': (_I, [_P, _P, _P, _I, _P, _I, _I, _I, _LL, _P, _P]),
    'ggp_reconstruct_stats_f32': (_I, [_P, _P, _P, _I, _P, _I, _P, _I, _I, _I, _LL, _D, _P, _P, _P, _P]),
    'ggp_errstats_workspace_bytes': (_LL, [_I, _LL]),
    'ggp_reconstruct_errstats_f32': (_I, [_P, _P, _P, _I, _P, _I, _P, _I, _I, _I, _LL, _D, _P, _F, _P, _P, _P, _P, _P, _LL, _P]),
    'ggp_reconstruct_stats_supported': (_I, [_I, _I, _D]),
    'ggp_reconstruct_quantiles_f32': (_I, [_P, _P, _P, _I, _P, _I, _P, _I, _I, _I, _LL, C.POINTER(_D), _I, _P, _P, _P]),
    'ggp_fields_errstats_f32': (_I, [_P, _P, _P, _P, _I, _LL, _F, _P, _P, _LL, _P]),
    'ggp_chain_diag_workspace_bytes': (_LL, [_I, _I, _I]),
    'ggp_chain_diag_f64': (_I, [_P, _I, _I, _I, _LL, _LL, _LL, _P, _P, _P, _P, _LL, _P]),
    'ggp_sobol_stats_f64': (_I, [_P, _P, _P, _I, _I, _I, _P, _LL, _I, _I, _I, _P, _P, _P]),
    'ggp_gp_sens_workspace_bytes': (_LL, [_I, _I, _I, _I, _I]),
    'ggp_gp_sens_f64': (_I, [_P, _I, _I, _P, _P, _I, _I, _I, _P, _P, _P, _LL, _P]),
    'ggp_main_effects_f64': (_I, [_P, _I, _I, _P, _P, _I, _I, _I, _P, _I, _P, _P, _LL, _P]),
    'ggp_rsvd_workspace_bytes': (_LL, [_I]),
    'ggp_rsvd_sketch_f32': (_I, [_P, _I, _LL, _P, _I, _P, _P, _LL, _P]),
    'ggp_rsvd_xty_f32': (_I, [_P, _I, _LL, _P, _I, _P, _P]),
    'ggp_rsvd_tc_workspace_bytes': (_LL, [_I]),
    'ggp_rsvd_sketch_tc_f32': (_I, [_P, _I, _LL, _P, _I, _P, _P, _LL, _P]),
    'ggp_rsvd_xty_tc_f32': (_I, [_P, _I, _LL, _P, _I, _P, _P]),
    'ggp_colstats_f32': (_I, [_P, _LL, _I, _LL, _I, _I, _F, _P, _P, _P]),
    'ggp_standardize_f32': (_I, [_P, _LL, _I, _LL, _I, _P, _LL, _P, _LL, _P, _P]),
    'ggp_project_workspace_bytes': (_LL, [_I, _I]),
    'ggp_project_f32': (_I, [_P, _I, _LL, _P, _I, _P, _P, _LL, _P]),
}


def load():
    """Load the shared library (once).  Raises GgpError if it is missing: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GgpError('libgladsgp_b200.so not found at %s -- run `python -c "import __graft_entry__ as g; '
                       'g.build()"` (needs nvcc); there is no CPU fallback' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header / library mismatch
        fn.restype = res
        fn.argtypes = args
    if lib.ggp_sizeof_mcmc_args() != C.sizeof(McmcArgs):
        raise GgpError('ggp_mcmc_args layout mismatch between _lib.py and the library')
    _lib = lib
    return lib


def check(rc, what=''):
    if rc != 0:
        msg = load().ggp_last_error_string().decode()
        raise GgpError('%s failed (%d): %s' % (what, rc, msg))


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise GgpError('gladsgp_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback')
    return torch


def ptr(t):
    """Device (or host) pointer of a torch tensor / None."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
