"""ctypes binding of libdctp.so - the only route from Python to the scoring kernels.

Mirrors include/dctp.h one to one.  Loading fails loudly: a missing library or a missing
CUDA device is an error, never a reason to compute on the CPU.
"""
import ctypes
import os

from .build import LIB_PATH

PATH_AUTO, PATH_UMMA, PATH_SIMT, PATH_TMEM, PATH_LARGE, PATH_STACK, PATH_KRON = 0, 1, 2, 3, 4, 5, 6
PATHS = {'auto': PATH_AUTO, 'umma': PATH_UMMA, 'simt': PATH_SIMT, 'tmem': PATH_TMEM, 'large': PATH_LARGE, 'stack': PATH_STACK, 'kron': PATH_KRON}

OP_DCT2, OP_RANK, OP_RANK_SQ, OP_DCT3 = 0, 1, 2, 3
OPS = {'dct2': OP_DCT2, 'rank': OP_RANK, 'rank_sq': OP_RANK_SQ, 'dct3': OP_DCT3}

OK, E_INVALID, E_CUDA, E_UNSUPPORTED, E_DEVICE = 0, -1, -2, -3, -4

DTYPE_F32, DTYPE_BF16, DTYPE_F16 = 0, 1, 2


def dtype_code(dtype):
    """DCTP_DTYPE_* of a torch dtype the score entries read (fp32, bf16, fp16), None for any other."""
    import torch
    return {torch.float32: DTYPE_F32, torch.bfloat16: DTYPE_BF16, torch.float16: DTYPE_F16}.get(dtype)

_c = ctypes
_SIGNATURES = {
    'dctp_version': (_c.c_int, []),
    'dctp_last_error': (_c.c_char_p, []),
    'dctp_init': (_c.c_int, []),
    'dctp_shutdown': (_c.c_int, []),
    'dctp_prepare': (_c.c_int, [_c.c_int, _c.c_int]),
    'dctp_score_accum': (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int,
                                    _c.c_longlong, _c.c_longlong, _c.c_longlong,
                                    _c.c_int, _c.c_int,
                                    _c.c_void_p, _c.c_void_p, _c.c_void_p,
                                    _c.c_int, _c.c_void_p]),
    'dctp_score_accum_ex': (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_int,
                                       _c.c_longlong, _c.c_longlong, _c.c_longlong,
                                       _c.c_int, _c.c_int,
                                       _c.c_void_p, _c.c_void_p, _c.c_void_p,
                                       _c.c_int, _c.c_void_p]),
    'dctp_score_accum_multi': (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p]),
    'dctp_score_accum_multi_ex': (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p]),
    'dctp_score_op': (_c.c_int, [_c.c_int, _c.c_void_p, _c.c_int, _c.c_int, _c.c_int,
                                 _c.c_longlong, _c.c_longlong, _c.c_longlong,
                                 _c.c_int, _c.c_int, _c.c_void_p, _c.c_void_p, _c.c_void_p]),
    'dctp_finalize': (_c.c_int, [_c.c_void_p, _c.c_double, _c.c_void_p, _c.c_int, _c.c_void_p]),
    'dctp_topk_segmented': (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_int,
                                       _c.c_void_p, _c.c_void_p, _c.c_void_p]),
    'dctp_gather_weight': (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int,
                                      _c.c_void_p, _c.c_int, _c.c_void_p, _c.c_void_p]),
    'dctp_check': (_c.c_int, [_c.c_void_p]),
    'dctp_score_host': (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_int, _c.c_int, _c.c_int,
                                   _c.c_void_p, _c.c_int]),
    'dctp_path_for': (_c.c_int, [_c.c_int, _c.c_int, _c.c_longlong]),
    'dctp_occupancy': (_c.c_int, [_c.c_int, _c.c_int]),
    'dctp_launch_count': (_c.c_longlong, []),
    'dctp_last_kernel': (_c.c_char_p, []),
    'dctp_sm_count': (_c.c_int, []),
}
EXPORTS = tuple(_SIGNATURES)


class Site(_c.Structure):
    """dctp_site of include/dctp.h: one dense activation of a multi-site launch (x: of the call's dtype)."""
    _fields_ = [('x', _c.c_void_p), ('accum', _c.c_void_p), ('B', _c.c_int), ('c_count', _c.c_int)]


class DctpError(RuntimeError):
    def __init__(self, code, text):
        super().__init__('libdctp error %d: %s' % (code, text))
        self.code = code


_lib = None


def load():
    """dlopen libdctp.so (built in-tree by dct_pruning_b200.build) and type its entry points."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError('libdctp.so not found at %s: run `python -c "import __graft_entry__ as g; g.build()"` '
                          '(or python -m dct_pruning_b200.build); there is no CPU fallback' % LIB_PATH)
    lib = ctypes.CDLL(os.environ.get('DCTP_LIB', LIB_PATH))     # (DCTP_LIB: an alternative build, for A/B measurements)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = the .so is stale w.r.t. include/dctp.h
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def check(code):
    if code != OK:
        raise DctpError(code, load().dctp_last_error().decode('utf-8', 'replace'))
    return code


def ptr(t):
    """Device/host address of a torch tensor (or None)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def current_stream():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
