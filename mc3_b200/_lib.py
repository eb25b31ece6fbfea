"""ctypes binding of libmc3b200.so (include/mc3b200.h).

The product has no CPU fallback: if the shared library is missing, or a call
fails (no GPU, CUDA error, bad argument), an exception is raised.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIBPATH = os.environ.get('MC3B_LIBPATH') or os.path.join(HERE, 'libmc3b200.so')

OK, ERR_ARG, ERR_CUDA = 0, 1, 2
F64, F32 = 0, 1
MRW, DEMC, SNOOKER = 0, 1, 2
SAMPLERS = {'mrw': MRW, 'demc': DEMC, 'snooker': SNOOKER}
MAX_PARS = 32
MAX_INPUTS = 4                    # MC3B_MAX_INPUTS: per-point inputs of a user model
GUARD_RECORDS = 64                # MC3B_GUARD_RECORDS: slots of the moment form's guard record ring

c_i64, c_i32, c_int = ctypes.c_int64, ctypes.c_int32, ctypes.c_int
c_vp, c_dbl = ctypes.c_void_p, ctypes.c_double


class Mc3bError(RuntimeError):
    pass


class SamplerStruct(ctypes.Structure):
    """mc3b_sampler_t -- field order must match include/mc3b200.h."""
    _fields_ = [
        ('nchains', c_i64), ('chain0', c_i64), ('nlocal', c_i64),
        ('npars', c_i32), ('nfree', c_i32), ('sampler', c_i32), ('reflect', c_i32),
        ('ifree', c_vp), ('pstep', c_vp), ('pmin', c_vp), ('pmax', c_vp),
        ('params0', c_vp), ('prior', c_vp), ('priorlow', c_vp), ('priorup', c_vp),
        ('gamma', c_dbl), ('fepsilon', c_dbl), ('seed', ctypes.c_uint64),
        ('X', c_vp), ('chisq_cur', c_vp), ('Z', c_vp), ('log_post', c_vp),
        ('zchain', c_vp), ('zlen', c_i64), ('M0', c_i64),
        ('nextp', c_vp), ('mrfactor', c_vp), ('u', c_vp), ('inb', c_vp),
        ('naccept', c_vp), ('outbounds', c_vp), ('best_chisq', c_vp),
        ('best_x', c_vp), ('best_gen', c_vp),
        ('gen_dev', c_vp), ('thinning', c_i64),
        ('X_peers', c_vp), ('Z_peers', c_vp), ('world', c_i32), ('rank', c_i32),
        ('F_peers', c_vp),
    ]


class BatchStruct(ctypes.Structure):
    """mc3b_batch_t."""
    _fields_ = [('nproblems', c_i64), ('problems', c_vp), ('offsets', c_vp),
                ('x', c_vp), ('data', c_vp), ('invsig', c_vp), ('status', c_vp)]


class SpectralStruct(ctypes.Structure):
    """mc3b_spectral_t."""
    _fields_ = [('table', c_vp), ('w1', c_dbl), ('w2', c_dbl), ('delta', c_dbl), ('xc', c_dbl),
                ('n1', c_i32), ('n2', c_i32), ('order', c_i32)]


class MomentStruct(ctypes.Structure):
    """mc3b_moment_t."""
    _fields_ = [('folded', c_vp), ('tiles', c_vp), ('c0ref', c_dbl), ('slref', c_dbl),
                ('d2tot', c_dbl), ('amp_max', c_dbl), ('xlo', c_dbl), ('xhi', c_dbl),
                ('guard_hits', c_vp), ('layout', c_i32), ('spectral', ctypes.POINTER(SpectralStruct)),
                ('record', c_vp)]


class ChisqOpts(ctypes.Structure):
    """mc3b_chisq_opts_t."""
    _fields_ = [('plan_chains', c_i64), ('uniform_sigma', c_i32), ('advance', c_i32),
                ('fuse', ctypes.POINTER(SamplerStruct)), ('fuse_done', c_vp),
                ('c_off', c_i64), ('gen', c_i64), ('zrow0', c_i64), ('folded', c_vp), ('work', c_vp),
                ('moment', ctypes.POINTER(MomentStruct)), ('tile_x', c_vp), ('dx', c_dbl),
                ('ntiles', c_i64)]


class UserModelDesc(ctypes.Structure):
    """mc3b_user_model_desc_t."""
    _fields_ = [('nmodel', c_int), ('ninputs', c_int), ('nconst', c_int), ('nwork', c_int), ('dtype', c_int)]


FOLD_WORK = 27                    # MC3B_FOLD_WORK


class DrawsStruct(ctypes.Structure):
    """mc3b_draws_t."""
    _fields_ = [('normal', c_vp), ('a', c_vp), ('b', c_vp), ('iz', c_vp),
                ('usj', c_vp), ('gs', c_vp), ('u', c_vp)]


_SIGS = {
    # name: (restype, argtypes)
    'mc3b_version': (c_int, []),
    'mc3b_last_error': (ctypes.c_char_p, []),
    'mc3b_device_sms': (c_int, []),
    'mc3b_model_chisq_plan': (c_int, [c_i64, c_i64, c_int, ctypes.POINTER(c_int)]),
    'mc3b_model_chisq_plan_kind': (c_int, [c_int, c_i64, c_i64, c_int, ctypes.POINTER(c_int)]),
    'mc3b_model_chisq_splits': (c_int, [c_i64, c_i64, c_int, ctypes.POINTER(c_i64), c_int,
                                        ctypes.POINTER(c_int)]),
    'mc3b_model_chisq': (c_int, [c_int, c_int, c_vp, c_i64, c_i64, c_int, c_vp,
                                 c_vp, c_vp, c_i64, c_vp, c_i64, c_int, c_vp]),
    'mc3b_model_chisq_ex': (c_int, [c_int, c_int, c_vp, c_i64, c_i64, c_int, c_vp,
                                    c_vp, c_vp, c_i64, c_vp, c_i64, c_int,
                                    ctypes.POINTER(ChisqOpts), c_vp]),
    'mc3b_fold_data': (c_int, [c_vp, c_i64, c_vp, c_vp]),
    'mc3b_moment_finish': (c_int, [ctypes.POINTER(MomentStruct), c_vp, c_i64, c_int, c_i64, c_vp, c_i64, c_int,
                                   c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'mc3b_moment_prepare': (c_int, [c_vp, c_i64, c_dbl, c_dbl, c_vp, c_dbl, c_dbl, c_int, c_vp, c_vp, c_vp]),
    'mc3b_spectral_size': (c_int, [c_int, c_int, c_int, ctypes.POINTER(c_i64)]),
    'mc3b_spectral_prepare': (c_int, [c_vp, c_vp, c_i64, c_dbl, c_dbl, ctypes.POINTER(SpectralStruct), c_vp]),
    'mc3b_model_eval': (c_int, [c_int, c_vp, c_i64, c_i64, c_int, c_vp, c_i64,
                                c_vp, c_vp]),
    'mc3b_user_model_compile': (c_int, [ctypes.c_char_p, ctypes.c_char_p, c_int, c_int, c_vp, c_i64,
                                        ctypes.POINTER(c_i64), ctypes.c_char_p, c_i64]),
    'mc3b_user_model_load': (c_int, [ctypes.c_char_p, c_i64, c_int, c_int, ctypes.POINTER(c_vp)]),
    'mc3b_user_model_free': (c_int, [c_vp]),
    'mc3b_user_model_chisq_ex': (c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64,
                                         c_int, ctypes.POINTER(ChisqOpts), c_vp]),
    'mc3b_user_model_eval': (c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp]),
    'mc3b_user_model_compile_ex': (c_int, [ctypes.c_char_p, ctypes.c_char_p, c_int, c_int, c_int, c_vp, c_i64,
                                           ctypes.POINTER(c_i64), ctypes.c_char_p, c_i64]),
    'mc3b_user_model_load_ex': (c_int, [ctypes.c_char_p, c_i64, c_int, c_int, c_int, ctypes.POINTER(c_vp)]),
    'mc3b_user_model_chisq_inputs': (c_int, [c_vp, c_vp, c_i64, c_i64, ctypes.POINTER(c_vp), c_int, c_vp, c_vp,
                                             c_i64, c_vp, c_i64, c_int, ctypes.POINTER(ChisqOpts), c_vp]),
    'mc3b_user_model_eval_inputs': (c_int, [c_vp, c_vp, c_i64, c_i64, ctypes.POINTER(c_vp), c_int, c_i64, c_vp,
                                            c_vp]),
    'mc3b_user_model_compile_desc': (c_int, [ctypes.c_char_p, ctypes.c_char_p, ctypes.POINTER(UserModelDesc), c_vp,
                                             c_i64, ctypes.POINTER(c_i64), ctypes.c_char_p, c_i64]),
    'mc3b_user_model_load_desc': (c_int, [ctypes.c_char_p, c_i64, ctypes.POINTER(UserModelDesc),
                                          ctypes.POINTER(c_vp)]),
    'mc3b_user_model_chisq_consts': (c_int, [c_vp, c_vp, c_i64, c_i64, ctypes.POINTER(c_vp), c_int, c_vp, c_int,
                                             c_vp, c_vp, c_i64, c_vp, c_i64, c_int, ctypes.POINTER(ChisqOpts), c_vp]),
    'mc3b_user_model_eval_consts': (c_int, [c_vp, c_vp, c_i64, c_i64, ctypes.POINTER(c_vp), c_int, c_vp, c_int,
                                            c_i64, c_vp, c_vp]),
    'mc3b_chisq_finish': (c_int, [c_vp, c_i64, c_int, c_i64, c_vp, c_i64, c_int,
                                  c_vp, c_vp, c_vp, c_vp, c_vp]),
    'mc3b_chisq_batch': (c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp]),
    'mc3b_residuals': (c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_i64,
                               c_vp, c_vp]),
    'mc3b_propose': (c_int, [ctypes.POINTER(SamplerStruct), c_i64, c_i64, c_i64,
                             c_i64, c_vp]),
    'mc3b_propose_replay': (c_int, [ctypes.POINTER(SamplerStruct),
                                    ctypes.POINTER(DrawsStruct), c_i64, c_i64, c_vp]),
    'mc3b_metropolis': (c_int, [ctypes.POINTER(SamplerStruct), c_vp, c_i64, c_int,
                                c_i64, c_i64, c_i64, c_i64, c_i64, c_vp]),
    'mc3b_peer_alloc': (c_int, [c_i64, ctypes.POINTER(c_vp), ctypes.c_char_p]),
    'mc3b_peer_open': (c_int, [ctypes.c_char_p, ctypes.POINTER(c_vp)]),
    'mc3b_peer_close': (c_int, [c_vp]),
    'mc3b_peer_free': (c_int, [c_vp]),
    'mc3b_host_device_pointer': (c_int, [c_vp, ctypes.POINTER(c_vp)]),
    'mc3b_pack_counters': (c_int, [ctypes.POINTER(SamplerStruct), c_vp, c_vp]),
    'mc3b_advance': (c_int, [ctypes.POINTER(SamplerStruct), c_vp]),
    'mc3b_run_small': (c_int, [ctypes.POINTER(SamplerStruct), c_int, c_int, c_vp, c_vp, c_vp,
                               c_i64, c_i64, c_i64, c_vp]),
    'mc3b_batch_init': (c_int, [ctypes.POINTER(BatchStruct), c_int, c_int, c_int, c_vp]),
    'mc3b_batch_run': (c_int, [ctypes.POINTER(BatchStruct), c_int, c_int, c_i64, c_i64, c_vp]),
    'mc3b_init_trials': (c_int, [ctypes.POINTER(SamplerStruct), c_int, c_i64, c_i64,
                                 c_vp, c_vp, c_vp]),
    'mc3b_log_prior': (c_int, [c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                               c_vp, c_vp]),
    'mc3b_gelman_rubin': (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_i64,
                                  c_i64, c_vp, c_vp, c_vp]),
    'mc3b_gelman_rubin_moments': (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_i64,
                                          c_i64, c_i64, c_i64, c_vp, c_vp]),
    'mc3b_gelman_rubin_psrf': (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_vp]),
    'mc3b_dwt_workspace': (c_i64, [c_i64, c_i64]),
    'mc3b_dwt_chisq': (c_int, [c_int, c_vp, c_i64, c_i64, c_int, c_int, c_vp, c_vp,
                               c_i64, c_vp, c_i64, c_vp, c_vp, c_vp]),
    'mc3b_user_model_dwt_chisq': (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, ctypes.POINTER(c_vp), c_int, c_vp,
                                          c_int, c_vp, c_i64, c_vp, c_vp, c_vp]),
    'mc3b_daub4': (c_int, [c_vp, c_i64, c_int, c_vp, c_vp, c_vp]),
    'mc3b_binrms_workspace': (c_i64, [c_i64, c_i64, c_i64]),
    'mc3b_binrms': (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp,
                            c_vp, c_vp, c_vp]),
    'mc3b_binarray': (c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]),
    'mc3b_hpd_workspace': (c_i64, [c_int]),
    'mc3b_hpd': (c_int, [c_vp, c_i64, c_int, c_dbl, c_vp, c_vp, c_vp]),
    'mc3b_fma_peak': (c_int, [c_int, c_i64, c_vp, ctypes.POINTER(c_dbl), c_vp]),
    'mc3b_fma_peak_variant': (c_int, [c_int, c_i64, c_vp, ctypes.POINTER(c_dbl), c_vp]),
}
EXPORTS = tuple(_SIGS)

_lib = None


def load():
    """Load the shared library (once) and declare every signature."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIBPATH):
        raise Mc3bError(
            f'{LIBPATH} not found: build it with `python -m mc3_b200.build` '
            '(there is no CPU fallback)')
    lib = ctypes.CDLL(LIBPATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)          # AttributeError = symbol missing
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def call(name, *args):
    """Call an int-returning entry point; raise Mc3bError on failure."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != OK:
        msg = lib.mc3b_last_error().decode('utf-8', 'replace')
        raise Mc3bError(f'{name} failed (status {rc}): {msg}')
    return rc


def ptrs(ts):
    """Host array of the device pointers of torch tensors (the `xs` of the
    mc3b_user_model_*_inputs entry points)."""
    return (c_vp*len(ts))(*[t.data_ptr() for t in ts])


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def ld(t):
    """Row stride (in elements) of a 2-D row-major tensor; a single-row tensor
    may carry a meaningless stride, so fall back to its width."""
    return t.stride(0) if t.shape[0] > 1 else max(int(t.stride(0)), int(t.shape[1]))


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream
