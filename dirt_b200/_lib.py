"""ctypes binding of libdirt_b200.so (the C ABI declared in include/dirt_b200.h).

Takes the place of `tf.load_op_library(_lib_path + '/librasterise.so')` in the reference
(dirt/rasterise_ops.py:5-10).  Unlike the reference, a missing library is an error, not a warning:
there is no CPU or eager fallback behind this module.
"""
import ctypes
import os

from . import build as _build

_lib = None

ERR_BAD_SHAPE = -1
ERR_NULL_POINTER = -2
ERR_WORKSPACE_TOO_SMALL = -3
ERR_BAD_CHANNEL_GROUPS = -4
ERR_TOO_MANY_VERTICES = -5
ERR_CUDA = -6
ERR_MISALIGNED = -7
ERR_STALE_WORKSPACE = -8
BWD_SHARED_GEOMETRY = 1
BWD_SKIP_POSITION = 2
BWD_SKIP_COLOUR = 4
SHARED_BACKGROUND = 8
SHARED_COLOURS = 16
SHARED_FACES = 32


def lib():
    """The loaded library.  Raises RuntimeError when libdirt_b200.so has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get('DIRT_B200_LIB') or _build.SO_PATH   # the override serves A/B timing of prebuilt variants (profiles/kbench.py)
    if not os.path.exists(path):
        raise RuntimeError(
            'dirt_b200: %s is missing; rasterisation is unavailable. Build it with '
            '`python -m dirt_b200.build` (needs nvcc, sm_100a).' % path)
    L = ctypes.CDLL(path)
    vp, i, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t
    L.dirt_error_string.restype = ctypes.c_char_p
    L.dirt_error_string.argtypes = [i]
    L.dirt_abi_version.restype = i
    L.dirt_last_launch_count.restype = i
    L.dirt_workspace_bytes.restype = sz
    L.dirt_workspace_bytes.argtypes = [i] * 6
    L.dirt_workspace_bytes_min.restype = sz
    L.dirt_workspace_bytes_min.argtypes = [i] * 6
    L.dirt_rasterise_forward.restype = i
    L.dirt_rasterise_forward.argtypes = [vp] * 6 + [i] * 6 + [vp, sz, vp]
    L.dirt_rasterise_forward_ex.restype = i
    L.dirt_rasterise_forward_ex.argtypes = [vp] * 6 + [i] * 6 + [vp, sz, vp, i]
    L.dirt_rasterise_backward.restype = i
    L.dirt_rasterise_backward.argtypes = [vp] * 8 + [i] * 6 + [ctypes.POINTER(ctypes.c_int), i, i, vp, sz, vp]
    L.dirt_rasterise_backward_ex.restype = i
    L.dirt_rasterise_backward_ex.argtypes = [vp] * 8 + [i] * 6 + [ctypes.POINTER(ctypes.c_int), i, i, i, vp, sz, vp]
    L.dirt_workspace_status.restype = i
    L.dirt_workspace_status.argtypes = [vp, sz] + [i] * 6 + [vp]
    L.dirt_rasterise_visibility.restype = i
    L.dirt_rasterise_visibility.argtypes = [vp] * 4 + [i] * 5 + [vp, sz, vp]
    L.dirt_peer_exchange_bytes.restype = sz
    L.dirt_peer_exchange_bytes.argtypes = [i, ctypes.c_longlong]
    L.dirt_peer_exchange.restype = i
    L.dirt_peer_exchange.argtypes = [vp, vp, ctypes.POINTER(vp), ctypes.POINTER(vp), i, i, ctypes.c_longlong, ctypes.c_uint, vp]
    L.dirt_kernel_timer_enable.restype = i
    L.dirt_kernel_timer_enable.argtypes = [i]
    L.dirt_kernel_timer_elapsed_ms.restype = ctypes.c_float
    _lib = L
    return _lib


EXPORTED_SYMBOLS = ['dirt_error_string', 'dirt_abi_version', 'dirt_workspace_bytes', 'dirt_workspace_bytes_min', 'dirt_rasterise_forward',
                    'dirt_rasterise_forward_ex',
                    'dirt_rasterise_backward', 'dirt_rasterise_backward_ex', 'dirt_workspace_status',
                    'dirt_rasterise_visibility', 'dirt_peer_exchange_bytes', 'dirt_peer_exchange', 'dirt_last_launch_count',
                    'dirt_kernel_timer_enable', 'dirt_kernel_timer_elapsed_ms']


def error_string(code):
    return lib().dirt_error_string(int(code)).decode()


def check(code, what):
    """Map a C-ABI return code onto the exception the reference op would raise."""
    if code == 0:
        return
    msg = '%s: %s' % (what, error_string(code))
    if code in (ERR_BAD_SHAPE, ERR_BAD_CHANNEL_GROUPS, ERR_TOO_MANY_VERTICES, ERR_NULL_POINTER, ERR_MISALIGNED):
        raise ValueError(msg)  # errors::InvalidArgument in the reference
    raise RuntimeError(msg)
