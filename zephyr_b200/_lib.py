"""ctypes binding of the C ABI declared in include/zephyr_b200.h.

The library is the hand-written sm_100a CUDA build ``zephyr_b200/libzephyr_b200.so``
(``python -m zephyr_b200.build``).  There is no CPU fallback: if the library is missing or no
CUDA device is visible, :func:`get_lib` raises.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libzephyr_b200.so')

HZ_OK, HZ_EINVAL, HZ_EDIM, HZ_ENOMEM, HZ_ECUDA, HZ_ESINGULAR, HZ_ESTATE, HZ_ENOTIMPL, HZ_EACCURACY = range(9)
HZ_C128, HZ_C64 = 0, 1
HZ_DISC_MINIZEPHYR, HZ_DISC_EURUS = 0, 1
HZ_OP_N, HZ_OP_T, HZ_OP_H = 0, 1, 2

_vp, _i64, _i32, _f64, _int = C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_int

# name -> (restype, argtypes); must list every symbol include/zephyr_b200.h declares
SIGNATURES = {
    'hz_version': (C.c_char_p, []),
    'hz_last_error': (C.c_char_p, [_vp]),
    'hz_create': (_int, [C.POINTER(_vp), _int, _int, _int, _i64, _i64, _f64, _f64, _int, _f64, C.POINTER(_i32), _vp]),
    'hz_destroy': (_int, [_vp]),
    'hz_set_stream': (_int, [_vp, _vp]),
    'hz_set_model': (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _int]),
    'hz_assemble': (_int, [_vp, _f64, _f64, _f64, _f64]),
    'hz_get_coefficients': (_int, [_vp, _vp]),
    'hz_set_coefficients': (_int, [_vp, _vp]),
    'hz_factor': (_int, [_vp, _i64]),
    'hz_has_factors': (_int, [_vp, C.POINTER(_i32)]),
    'hz_free_factors': (_int, [_vp]),
    'hz_factor_bytes': (_int, [_vp, C.POINTER(_i64)]),
    'hz_get_block_inverse': (_int, [_vp, _i64, _vp]),
    'hz_solve': (_int, [_vp, _vp, _i64, _f64, _f64, _int, _i64, _i64, _int, C.POINTER(_f64)]),
    'hz_solve_op': (_int, [_vp, _int, _vp, _i64, _f64, _f64, _int, _i64, _i64, _int, C.POINTER(_f64)]),
    'hz_synchronize': (_int, [_vp]),
    'hz_last_probe': (_int, [_vp, C.POINTER(_f64)]),
    'hz_profile': (_int, [_vp, _int, C.POINTER(_f64)]),
    'hz_launch_count': (_int, [C.POINTER(_i64)]),
    'hz_newton_stats_get': (_int, [C.POINTER(_i64)]),
    'hz_factor_graph_info': (_int, [_vp, C.POINTER(_i64)]),
    'hz_factor_resident_bytes': (_int, [_vp, C.POINTER(_i64)]),
    'hz_set_option': (_int, [_vp, C.c_char_p, _f64]),
    'hz_get_trace': (_int, [_vp, _vp, _i64, C.POINTER(_i64), C.POINTER(_i64)]),
    'hz_scatter_coo': (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _f64, _f64, _vp]),
    'hz_nearest_index': (_int, [_i64, _i64, _f64, _f64, _f64, _f64, _vp, _i64, _vp, _vp]),
    'hz_kaiser_taps': (_int, [_i64, _i64, _f64, _f64, _f64, _f64, _int, C.POINTER(_i32), _vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    'hz_spmm_csr': (_int, [_i64, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _i64, _i64, _int, _vp]),
    'hz_spmm_percol': (_int, [_int, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _i64, _vp]),
    'hz_spmm_percol_c64': (_int, [_int, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _i64, _vp]),
    'hz_gradient': (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    'hz_misfit': (_int, [_vp, _vp, _i64, _f64, _vp, _vp, _vp]),
    'hz_stencil_xcorr': (_int, [_vp, _vp, _i64, _i64, _i64, _vp, _vp]),
    'hz_assemble_vjp': (_int, [_vp, _vp, _vp, _vp, _vp]),
    'hz_stencil_apply': (_int, [_vp, _vp, _i64, _i64, _i64, _f64, _f64, _vp, _vp]),
    'hz_assemble_jvp': (_int, [_vp, _vp, _vp, _vp, _vp]),
    'hz_wavefield_lagcorr': (_int, [_vp, _i64, _i64, _i64, _vp, _vp]),
    'hz_pseudo_hessian': (_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    'hz_wavefield_lagcorr4': (_int, [_vp, _i64, _i64, _i64, _vp, _vp]),
    'hz_gauss_newton_diag': (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'hz_scatter_coo_c64': (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _f64, _f64, _vp]),
    'hz_spmm_csr_c64': (_int, [_i64, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _i64, _i64, _int, _vp]),
    'hz_gradient_c64': (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    'hz_misfit_c64': (_int, [_vp, _vp, _i64, _f64, _vp, _vp, _vp]),
    'hz_cgemm_tf32': (_int, [_i64, _i64, _i64, _f64, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _int]),
    'hz_zgemm': (_int, [_i64, _i64, _i64, _f64, _vp, _i64, _vp, _i64, _int, _vp, _i64, _int, _vp]),
    'hz_zgemm_op': (_int, [_i64, _i64, _i64, _f64, _vp, _i64, _int, _vp, _i64, _int, _vp, _i64, _int, _int, _vp]),
}


class HzError(RuntimeError):
    pass


def bind(path):
    """dlopen `path` and attach the signatures; raises if a declared symbol is missing."""
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)              # AttributeError => symbol not exported
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = None


def get_lib():
    """The CUDA library; loud failure when it (or a GPU) is absent."""
    global _lib
    if _lib is None:
        import torch
        if not torch.cuda.is_available():
            raise HzError('zephyr_b200 needs a CUDA device (built for sm_100a); there is no CPU fallback')
        if not os.path.exists(LIB_PATH):
            raise HzError('%s is missing: build it with `python -m zephyr_b200.build`' % LIB_PATH)
        _lib = bind(LIB_PATH)
    return _lib


def torch_device(index=None):
    import torch
    return torch.device('cuda', torch.cuda.current_device() if index is None else int(index))


def current_stream_ptr(device):
    import torch
    if device.type != 'cuda':
        return None
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


_EXC = {HZ_EINVAL: ValueError, HZ_EDIM: ValueError, HZ_ENOMEM: MemoryError, HZ_ECUDA: HzError,
        HZ_ESINGULAR: np.linalg.LinAlgError, HZ_ESTATE: HzError, HZ_ENOTIMPL: NotImplementedError,
        HZ_EACCURACY: np.linalg.LinAlgError}


def check(rc, handle=None):
    """Map a status code to the exception type the reference would raise (SURVEY.md 8(b))."""
    if rc == HZ_OK:
        return
    msg = get_lib().hz_last_error(handle)
    msg = msg.decode() if msg else 'zephyr_b200 error %d' % rc
    raise _EXC.get(rc, HzError)(msg)


def trans_op(trans):
    """``trans`` of scipy's ``SuperLU.solve`` ('N', 'T', 'H') -> HZ_OP_N / HZ_OP_T / HZ_OP_H."""
    try:
        return {'N': HZ_OP_N, 'T': HZ_OP_T, 'H': HZ_OP_H}[trans]
    except (KeyError, TypeError):
        raise ValueError("trans must be 'N', 'T' or 'H', not %r" % (trans,))


def panel_fn(name, c64):
    """Panel-typed entry point: `name` for complex128 panels, `name_c64` for complex64 panels."""
    return getattr(get_lib(), name + ('_c64' if c64 else ''))


def ptr(t):
    """Device (or pinned-host) pointer of a torch tensor / numpy array as c_void_p; None passes NULL."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return C.c_void_p(t.ctypes.data)
    return C.c_void_p(t.data_ptr())
