"""ctypes binding of libqce_b200.so (include/qce_b200.h).  No fallback: if the library is missing
or no B200 is visible, the hot-path calls raise."""
import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, 'libqce_b200.so')

MODE_ALL, MODE_TOP1, MODE_TOPN, MODE_CUMPROB = 0, 1, 2, 3
PREC_FP64, PREC_TC = 0, 1
FLAG_TOP1_EXP_ARGMAX = 1
ERR_UNSUPPORTED = -3

_lib = None

_SIGS = {
    'qce_abi_version': (C.c_int, []),
    'qce_last_error_string': (C.c_char_p, []),
    'qce_launch_count': (C.c_int64, []),
    'qce_device_ok': (C.c_int, []),
    'qce_last_fix_count': (C.c_int64, [C.c_void_p]),
    'qce_host_staging_release': (None, []),
    'qce_estimate_host_codes': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_int]),
    'qce_quantizer_create': (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    'qce_quantizer_destroy': (None, [C.c_void_p]),
    'qce_quantize': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    'qce_observe_quantize': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_double,
                                       C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    'qce_model_create': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    'qce_model_destroy': (None, [C.c_void_p]),
    'qce_model_set_params': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_double]),
    'qce_estimate': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_int,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'qce_pipeline': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_double,
                               C.c_int64, C.c_int, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_void_p]),
    'qce_format_pilots': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    'qce_estimate_formatted': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    'qce_circ_model_create': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    'qce_circ_model_destroy': (None, [C.c_void_p]),
    'qce_circ_model_set_params': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'qce_circ_estimate': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    'qce_circ_estimate_prec': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_int,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'qce_mfa_model_create': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    'qce_mfa_model_destroy': (None, [C.c_void_p]),
    'qce_mfa_model_set_params': (C.c_int, [C.c_void_p] * 9),
    'qce_mfa_estimate': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    'qce_rate_model_create': (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    'qce_rate_model_destroy': (None, [C.c_void_p]),
    'qce_rate_model_set_params': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'qce_rate_accumulate': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p]),
    'qce_estimate_host': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_int,
                                    C.c_void_p]),
    'qce_circ_estimate_host': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_int,
                                         C.c_void_p]),
    'qce_mfa_estimate_host': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_void_p]),
}
EXPORTS = tuple(_SIGS)


class QceError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f'qce_b200 error {status}: {msg}')
        self.status = status


def load():
    """Load the shared library (once) and set the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f'{LIB_PATH} is missing: build it with `python -m quantized_channel_estimation_b200.build` '
                           '(__graft_entry__.build()); there is no CPU fallback for the hot path')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.qce_abi_version() != 1:
        raise RuntimeError('libqce_b200.so ABI mismatch')
    _lib = lib
    return lib


def check(status):
    if status != 0:
        raise QceError(status, load().qce_last_error_string().decode())


def require_device():
    lib = load()
    if not lib.qce_device_ok():
        raise RuntimeError('qce_b200: no B200 (sm_100) CUDA device visible; the estimate/quantise kernels have no CPU fallback')
    return lib


def launch_count():
    return int(load().qce_launch_count())
