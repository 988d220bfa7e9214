"""ctypes binding of the C ABI declared in include/cimrgp.h (cimrgp_b200/libcimrgp.so).

There is no CPU fallback: if the shared library is missing the import fails, and every compute entry
point fails with MRGP_ENODEVICE when no sm_100 device is present."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libcimrgp.so')

COMM_BLOB_BYTES = 128
ABI_VERSION = 5
MODE_CI, MODE_FI = 0, 1
OK, EINVAL, ENODEVICE, ECUDA, ESTATE, ENOMEM = 0, -1, -2, -3, -4, -5

# field ids (include/cimrgp.h)
F_L, F_LAMBDA, F_SPECTRAL, F_PHI2SUM = 1, 2, 3, 4
F_SCALE_PRECISION, F_ZETA, F_YTILDE, F_NOISE_SHAPE, F_NOISE_SCALE, F_BIAS_PRECISION = 10, 11, 12, 13, 14, 15
F_A, F_M2, F_CM2, F_NOISE_MEAN, F_NOISE_LOG_MEAN, F_BIAS_MEAN, F_BIAS_VAR = 20, 21, 22, 23, 24, 25, 26
F_FBAR, F_FVAR, F_YVAR, F_PHASE_B_SUMS, F_A_PREV, F_BIAS_PREV = 27, 28, 29, 30, 31, 32
F_AXIS_B, F_AXIS_KAPPA, F_AXIS_RHO, F_AXIS_LOGC, F_AXIS_COV = 40, 41, 42, 43, 44
F_ARD_SHAPE, F_ARD_SCALE, F_ARD_MEAN, F_ARD_LOG_MEAN, F_OMEGA, F_LOG_OMEGA_HAT = 45, 46, 47, 48, 49, 50
F_OMEGA_ITERS = 51
F_FUSED_GUARD = 55


class Config(C.Structure):
    _fields_ = [('abi_version', C.c_int32), ('mode', C.c_int32), ('n_samples', C.c_int64), ('dx', C.c_int32),
                ('dy', C.c_int32), ('n_basis', C.c_int32), ('n_layers', C.c_int32),
                ('noise_region_specific', C.c_int32), ('bias_region_specific', C.c_int32), ('device', C.c_int32),
                ('n_ctas', C.c_int32), ('sample_begin', C.c_int64), ('sample_end', C.c_int64)]


class MrgpError(RuntimeError):
    def __init__(self, code, message):
        RuntimeError.__init__(self, 'cimrgp error %d: %s' % (code, message))
        self.code = code


_P = C.c_void_p
_D = C.POINTER(C.c_double)
_I64PP = C.POINTER(C.POINTER(C.c_int64))

# name -> (restype, argtypes); every symbol include/cimrgp.h declares
SIGNATURES = {
    'mrgp_abi_version': (C.c_int, []),
    'mrgp_create': (C.c_int, [C.POINTER(Config), _I64PP, C.POINTER(C.c_int32), C.POINTER(_P)]),
    'mrgp_destroy': (None, [_P]),
    'mrgp_last_error': (C.c_char_p, [_P]),
    'mrgp_workspace_bytes': (C.c_size_t, [_P]),
    'mrgp_bind_workspace': (C.c_int, [_P, _P, C.c_size_t]),
    'mrgp_set_stream': (C.c_int, [_P, _P]),
    'mrgp_set_data': (C.c_int, [_P, _P, _P]),
    'mrgp_set_data_host': (C.c_int, [_P, _P, _P]),
    'mrgp_set_observations': (C.c_int, [_P, _P]),
    'mrgp_set_observations_host': (C.c_int, [_P, _P]),
    'mrgp_prefetch_observations_host': (C.c_int, [_P, _P]),
    'mrgp_prefetch_sync': (C.c_int, [_P]),
    'mrgp_set_fused': (C.c_int, [_P, C.c_int32]),
    'mrgp_set_spectral': (C.c_int, [_P, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_double]),
    'mrgp_build_basis': (C.c_int, [_P, C.c_int32, C.c_double, _D]),
    'mrgp_init_state': (C.c_int, [_P, C.c_double, C.c_double]),
    'mrgp_get_state': (C.c_int, [_P, C.c_int32, C.c_int32, _D, C.c_size_t]),
    'mrgp_set_state': (C.c_int, [_P, C.c_int32, C.c_int32, _D, C.c_size_t]),
    'mrgp_state_elems': (C.c_int64, [_P, C.c_int32, C.c_int32]),
    'mrgp_phase_a': (C.c_int, [_P, C.c_int32]),
    'mrgp_axis_update': (C.c_int, [_P, C.c_int32]),
    'mrgp_phase_b': (C.c_int, [_P, C.c_int32]),
    'mrgp_bias_noise': (C.c_int, [_P, C.c_int32]),
    'mrgp_set_adaptive_intervals': (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_double]),
    'mrgp_interval_failures': (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    'mrgp_learn_intervals': (C.c_int, [_P, C.c_int32]),
    'mrgp_sweep': (C.c_int, [_P, C.c_int32]),
    'mrgp_refresh_statistics': (C.c_int, [_P]),
    'mrgp_group_create': (C.c_int, [C.POINTER(_P), C.c_int32, _P, C.POINTER(_P)]),
    'mrgp_group_sweep': (C.c_int, [_P, C.c_int32]),
    'mrgp_group_observations_changed': (C.c_int, [_P]),
    'mrgp_group_launch_count': (C.c_int64, [_P]),
    'mrgp_group_synchronize': (C.c_int, [_P]),
    'mrgp_group_destroy': (None, [_P]),
    'mrgp_synchronize': (C.c_int, [_P]),
    'mrgp_elbo': (C.c_int, [_P, _D]),
    'mrgp_elbo_async': (C.c_int, [_P, _P, C.c_int32]),
    'mrgp_elbo_wait': (C.c_int, [_P, C.c_int32]),
    'mrgp_predict_mean': (C.c_int, [_P, _P, C.c_int64, _I64PP, C.c_int32, _P]),
    'mrgp_predict_var_indexed': (C.c_int, [_P, _P, C.c_int64, _I64PP, C.c_int32, _P]),
    'mrgp_predict_var': (C.c_int, [_P, _P, C.c_int64, _P]),
    'mrgp_comm_export': (C.c_int, [_P, C.c_void_p]),
    'mrgp_comm_bind': (C.c_int, [_P, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(C.c_int64)]),
    'mrgp_exchange': (C.c_int, [_P, C.c_int32, C.c_int32]),
    'mrgp_set_all_inputs_host': (C.c_int, [_P, _D]),
    'mrgp_launch_count': (C.c_int64, [_P]),
    'mrgp_cholesky_count': (C.c_int64, [_P]),
    'mrgp_batched_cholesky': (C.c_int, [_P, _P, C.c_int32, C.c_int64, _P]),
    'mrgp_fp64_probe': (C.c_int, [_P, C.c_int64, _P, C.POINTER(C.c_float)]),
    'mrgp_timeline_enable': (C.c_int, [_P, C.c_int32]),
    'mrgp_timeline_read': (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_float), C.c_int32]),
    'mrgp_plan_info': (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    'mrgp_plan_segments': (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int64)]),
    'mrgp_plan_pieces': (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    'mrgp_host_digamma': (C.c_double, [C.c_double]),
    'mrgp_host_matern_spectral': (C.c_double, [C.c_double, C.c_double, C.c_double, C.c_double]),
    'mrgp_host_bingham2': (None, [_D, _D, _D, _D, _D, _D, C.POINTER(C.c_int32)]),
    'mrgp_host_basis': (None, [C.c_double, C.c_double, C.c_int32, _D]),
    'mrgp_host_omega': (C.c_int, [_D, C.c_int32, _D, C.POINTER(C.c_int32)]),
}

_lib = None


def load():
    """dlopen the in-tree shared library (built by build.sh / __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError('%s is missing: run ./build.sh (nvcc, sm_100a). There is no CPU fallback.' % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        if lib.mrgp_abi_version() != ABI_VERSION:
            raise ImportError('ABI version mismatch')
        _lib = lib
    return _lib


def check(handle, rc):
    if rc != 0:
        msg = load().mrgp_last_error(handle)
        raise MrgpError(rc, msg.decode() if msg else '')


def offsets_arg(offsets):
    """list of int64 numpy arrays -> (int64** argument, keep-alive)."""
    import numpy as np
    arrs = [np.ascontiguousarray(o, dtype=np.int64) for o in offsets]
    ptrs = (C.POINTER(C.c_int64) * len(arrs))(*[a.ctypes.data_as(C.POINTER(C.c_int64)) for a in arrs])
    return ptrs, arrs
